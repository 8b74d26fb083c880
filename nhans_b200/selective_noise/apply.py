"""Drop-in mirror of N_HANS___Selective_Noise/apply.py on the B200 engine.

Same entry points, argument meaning and file side effects as the reference:
``apply_denoiser(mixedpath, negpath, save_to)`` (SN/apply.py:478-481), ``apply_snc(mixedpath, pospath,
negpath, save_to)`` (:339-472), ``recover_samples_from_spectrum`` (:189-204), ``handle_signals`` (:142-167),
``read_wav`` (:46-53), flags ``--input --neg --pos --output --compensate --ac`` (:29-35), plus the folder
mode the README advertises (README.md:59-66) and the ``main()`` the console script expects (setup.py:46).
All arithmetic runs in libnhans_b200.so on the GPU; there is no TensorFlow and no CPU fallback.

Differences from the reference, all deliberate (SURVEY.md F1/F2/F10): wav outputs are 16-bit PCM by
default (the north-star surface; ``--float32`` / ``out_format='float32'`` restores the reference's
float32 files), scaled back by the input peak that ``handle_signals`` divided out; a whole folder is
processed as one GPU batch."""
from __future__ import annotations

import argparse
import os
import sys

import numpy as np

from .. import weights as W
from ..session import get_engine
from ..wavio import FS, is_pcm16, normalise_host, read_wav, write_wav

Noise_Win = 200      # SN/apply.py:37
Mix_Win = 35         # SN/apply.py:38
VARIANT = W.SELECTIVE_NOISE
_SILENT = "Silent.wav"


class _Flags:        # the absl FLAGS of SN/apply.py:29-35
    input = "./audio_examples/mixed.wav"
    neg = "./audio_examples/game_noise.wav"
    pos = "./audio_examples/Silent.wav"
    output = "./audio_examples/denoised.wav"
    compensate = 0.0
    ac = False
    Fs = FS
    float32 = False


FLAGS = _Flags()


def handle_signals(mixedpath, noisepospath, noisenegpath):
    """SN/apply.py:142-163: (pos, neg, mixed) peak-normalised float32, the mixture trimmed to whole frames."""
    eng = get_engine(VARIANT)

    def norm(path, trim):
        x = read_wav(path)
        if is_pcm16(x):
            return eng.normalise([x], trim=trim)[0]
        y = normalise_host(x)                                      # stereo file: float64 mean, normalised on the host
        if trim and len(y) >= 400:
            y = y[:len(y) - (len(y) - 400) % 160]
        return y
    return norm(noisepospath, False), norm(noisenegpath, False), norm(mixedpath, True)


def _seq_sum(x):
    # the reference uses the Python builtin sum() over a float32 array (SN/apply.py:77-79): a sequential
    # accumulation that starts from int 0 and therefore runs in float64 under the numpy of its era
    return float(np.cumsum(np.asarray(x, np.float64))[-1]) if len(x) else 0.0


def _fit_noise(noise, n):
    # SN/apply.py:57-72: repeat the noise until it covers the speech, or cut it
    nse = noise
    while n - len(nse) > 0:
        nse = np.concatenate([nse, noise[:n - len(nse)]], axis=0)
    return nse[:n] if len(noise) > n else nse


def domixing(cleansamples, noisepossamples, noisenegsamples, snr_pos, snr_neg):
    """SN/apply.py:56-104 (host arithmetic, float32 arrays with float64 scalars like the reference)."""
    sig = np.asarray(cleansamples, np.float32)
    nse_pos = _fit_noise(np.asarray(noisepossamples, np.float32), len(sig))
    nse_neg = _fit_noise(np.asarray(noisenegsamples, np.float32), len(sig))
    psignal = _seq_sum(abs(sig) * abs(sig)) / sig.shape[0]
    pnoise_pos = _seq_sum(abs(nse_pos) * abs(nse_pos)) / nse_pos.shape[0]
    pnoise_neg = _seq_sum(abs(nse_neg) * abs(nse_neg)) / nse_neg.shape[0]
    K_pos = 1.0 if pnoise_pos == 0 else float(np.sqrt((psignal / pnoise_pos) * pow(10, -snr_pos / 10.0)))
    K_neg = 1.0 if pnoise_neg == 0 else float(np.sqrt((psignal / pnoise_neg) * pow(10, -snr_neg / 10.0)))
    noise_pos_scaled = np.float32(K_pos) * nse_pos
    noise_neg_scaled = np.float32(K_neg) * nse_neg
    mixed = sig + noise_pos_scaled + noise_neg_scaled
    mixed = mixed / np.float32(float(max(abs(mixed))) + 0.000001)
    d = np.float32(float(max(abs(mixed))) + 0.000001)          # the reference renormalises by the *normalised* mixture
    target = (sig + noise_pos_scaled) / d
    return mixed, target, K_pos, K_neg, noise_pos_scaled / d, noise_neg_scaled / d


_norm64 = normalise_host


def combine_signals(cleanpath, noisepospath, noisenegpath):
    """SN/apply.py:107-139: normalise the three recordings, trim the speech to whole frames, mix at 0 dB / 0 dB.
    -> (noise_pos_signal, noise_neg_signal, mixed, snr_pos, snr_neg)."""
    clean = _norm64(read_wav(cleanpath))
    pos = _norm64(read_wav(noisepospath))
    neg = _norm64(read_wav(noisenegpath))
    rem = (len(clean) - 400) % 160
    if rem != 0:
        clean = clean[:-rem]
    snr_pos = snr_neg = 0                                         # SNRs[1]
    mixed, _, _, _, pos_sig, neg_sig = domixing(clean, pos, neg, snr_pos, snr_neg)
    return pos_sig, neg_sig, mixed, np.array(snr_pos, np.int32), np.array(snr_neg, np.int32)


def apply_demo(speechpath, pospath, negpath, save_to):
    """SN/apply.py:212-337: mix speech with a positive and a negative noise on the fly, condition on the first
    200 frames of the scaled noises, process the mixture from frame 200 on.  Writes ``save_to`` and
    ``save_to[:-15] + 'mixed_demo.wav'`` (float32, like the reference)."""
    pos_sig, neg_sig, mixed, _, _ = combine_signals(speechpath, pospath, negpath)
    eng = get_engine(VARIANT)
    y, ymix = eng.enhance_demo(mixed, pos_sig, neg_sig, start=Noise_Win)
    write_wav(save_to, y)
    write_wav(save_to[:-15] + "mixed_demo.wav", ymix)
    return y, ymix


def recover_samples_from_spectrum(logspectrum_stft, spectrum_phase, save_to):
    """SN/apply.py:189-204: log-magnitude + phase -> samples (float32), written to ``save_to`` as float32 wav."""
    eng = get_engine(VARIANT)
    lm = np.ascontiguousarray(logspectrum_stft, np.float32)
    samples, _ = eng.istft(lm, spectrum_phase, np.array([0, lm.shape[0]], np.int64))
    if save_to:
        write_wav(save_to, samples)
    return samples


def _is_silent(path):
    return path is None or os.path.basename(path) == _SILENT


def _sibling(save_to, name):
    # the reference derives the extra outputs with save_to[:-12] (assumes '...denoised.wav', SN/apply.py:457)
    if save_to.endswith("denoised.wav"):
        return save_to[:-12] + name
    root, _ = os.path.splitext(save_to)
    return root + "_" + name


def _to_i16(f32, peak):
    v = np.rint(f32.astype(np.float32) * np.float32(peak + 0.000001))
    return np.clip(v, -32768, 32767).astype(np.int16)


def _emit(save_to, f32, peak, as_float32):
    write_wav(save_to, f32.astype(np.float32) if as_float32 else _to_i16(f32, peak))


def _post_mix_host(den, mixed, compensate, ac):
    # SN/apply.py:459-470 for the (rare) clips that take the float path
    removed = mixed - den
    with np.errstate(divide="ignore", invalid="ignore"):
        snr_est = float(np.mean(den.astype(np.float64) ** 2) / np.mean(removed.astype(np.float64) ** 2)) if len(den) else float("inf")
    factor = snr_est / 20.0 if ac else compensate
    if not np.isfinite(factor):
        factor = 0.0
    return removed, snr_est, (den + removed * np.float32(factor)).astype(np.float32)


def apply_snc_batch(mixedpaths, pospaths, negpaths, save_tos, compensate=None, ac=None, out_format=None):
    """apply_snc for many files in one GPU batch (folder mode).  pospaths entries may be None / Silent.wav: those
    utterances are conditioned on the all-zero Silent context (SN/apply.py:478-481), whatever the others use."""
    compensate = FLAGS.compensate if compensate is None else compensate
    ac = FLAGS.ac if ac is None else ac
    as_f32 = (FLAGS.float32 if out_format is None else out_format == "float32")
    eng = get_engine(VARIANT)
    mixes = [read_wav(p) for p in mixedpaths]
    negs = [read_wav(p) for p in negpaths]
    silent = [_is_silent(p) for p in pospaths]
    poss = [None if sil else read_wav(p) for p, sil in zip(pospaths, silent)]
    U = len(mixes)
    # int16 PCM clips go through the fused batch entry point; a clip set with a stereo file (float64 mean) takes the
    # float entry points one utterance at a time
    pcm = [u for u in range(U) if is_pcm16(mixes[u]) and is_pcm16(negs[u]) and (poss[u] is None or is_pcm16(poss[u]))]
    out = [None] * U
    if pcm:
        if all(silent[u] for u in pcm):
            pos_clips = None                                       # the engine's cached Silent.wav embedding
        else:
            zero = np.zeros(3 * FS, np.int16)                      # Silent.wav stand-in: >= 32240 samples of digital silence
            pos_clips = [zero if poss[u] is None else poss[u] for u in pcm]
        res = eng.enhance([mixes[u] for u in pcm], pos_clips, [negs[u] for u in pcm], want_f32=True, want_i16=False)
        # removed / snr_est / compensated (SN/apply.py:459-470) come from one fused GPU pass over the batch
        post = eng.postmix(res["out_offs"], compensate=compensate, ac=ac)
        for j, u in enumerate(pcm):
            out[u] = (res["f32"][j], post["mixed_processed"][j], post["removed"][j], float(post["snr_est"][j]), post["compensated"][j],
                      float(max(abs(mixes[u]))) if len(mixes[u]) else 0.0)
    for u in range(U):
        if out[u] is None:
            r = eng.enhance_float(mixes[u], poss[u], negs[u])
            removed, snr_est, comp = _post_mix_host(r["f32"], r["mixed_processed"], compensate, ac)
            out[u] = (r["f32"], r["mixed_processed"], removed, snr_est, comp, r["peak"])
    snrs = []
    for u, save_to in enumerate(save_tos):
        den, mixed, removed, snr_est, comp, peak = out[u]
        _emit(save_to, den, peak, as_f32)
        _emit(_sibling(save_to, "mixed_processed.wav"), mixed, peak, as_f32)
        _emit(_sibling(save_to, "removed.wav"), removed, peak, as_f32)
        print(snr_est)
        print("---------------------------")
        _emit(_sibling(save_to, "compensated.wav"), comp, peak, as_f32)
        snrs.append(snr_est)
    return snrs


def apply_snc(mixedpath, pospath, negpath, save_to):
    """SN/apply.py:339-472: selective noise suppression conditioned on a positive and a negative recording."""
    apply_snc_batch([mixedpath], [pospath], [negpath], [save_to])


def apply_denoiser(mixedpath, negpath, save_to):
    """SN/apply.py:478-481: pure denoising; the positive context is the all-zero Silent.wav, whose embedding
    is a per-model constant the engine caches."""
    apply_snc(mixedpath, None, negpath, save_to)


def _pairs(inp, pos, neg, out):
    """README.md:59-66 folder mode: files with identical names in the input / pos / neg folders."""
    names = sorted(f for f in os.listdir(inp) if f.lower().endswith(".wav"))
    os.makedirs(out, exist_ok=True)
    mixed, poss, negs, outs = [], [], [], []
    for n in names:
        npth = os.path.join(neg, n)
        if not os.path.exists(npth):
            sys.stderr.write("skipping %s: no --neg file of the same name\n" % n)
            continue
        mixed.append(os.path.join(inp, n))
        negs.append(npth)
        ppth = os.path.join(pos, n) if pos and os.path.isdir(pos) else None
        poss.append(ppth if ppth and os.path.exists(ppth) else None)
        outs.append(os.path.join(out, n[:-4] + "_denoised.wav"))
    return mixed, poss, negs, outs


# ---- live mode (--stream): raw PCM in, raw PCM out, through the engine's streaming entry points ----------------------
def add_stream_args(ap):
    ap.add_argument("--stream", action="store_true",
                    help="live mode: --input is raw s16le mono 16 kHz PCM ('-' = stdin), --output raw PCM ('-' = stdout), "
                         "s16le or f32le with --float32")
    ap.add_argument("--peak", type=int, default=32767, help="--stream: the int16 peak that scales the input and the output")
    ap.add_argument("--chunk-ms", type=int, default=100, help="--stream: largest read from the input, in ms of audio")


def check_stream_args(ap, a):
    if a.peak < 0:
        ap.error("--peak must not be negative")
    if a.chunk_ms < 1:
        ap.error("--chunk-ms must be at least 1")


def stream_context(ap, path, flag):
    """A context wav of a live stream: it must be int16 mono, the only form the int16 stream path conditions on exactly."""
    x = read_wav(path)
    if not is_pcm16(x):
        ap.error("%s %s: --stream needs an int16 mono context file (a stereo file is averaged in float64, which only the "
                 "batch path reproduces)" % (flag, path))
    return x


def pcm_bytes(x):
    """Raw little-endian bytes of int16 (s16le) or float32 (f32le) samples."""
    return np.asarray(x, x.dtype.newbyteorder("<")).tobytes()


def stream_pipe(step, inp, out, chunk_ms):
    """Feed raw s16le samples from `inp` ('-' = stdin) to step(samples, final) -> bytes and write what it returns to `out`
    ('-' = stdout), flushed after every step.  Each read takes what the pipe holds, at most one chunk, so a slow source is
    not held back; an odd trailing byte waits for the next read.  At EOF an empty final step flushes the stream."""
    fd = sys.stdin.fileno() if inp == "-" else os.open(inp, os.O_RDONLY)
    dst = sys.stdout.buffer if out == "-" else open(out, "wb")
    try:
        want, carry = 2 * (FS // 1000) * chunk_ms, b""
        while True:
            data = os.read(fd, want)
            if not data:
                break
            buf = carry + data
            n = len(buf) & ~1
            carry = buf[n:]
            if n:
                dst.write(step(np.frombuffer(buf[:n], "<i2").astype(np.int16), False))
                dst.flush()
        if carry:
            sys.stderr.write("ignoring an odd trailing byte at the end of the input\n")
        dst.write(step(np.zeros(0, np.int16), True))
        dst.flush()
    finally:
        if inp != "-":
            os.close(fd)
        if out != "-":
            dst.close()


def stream_denoiser(ap, a):
    """--stream: the compensated signal (denoised + removed * --compensate) of one live stream; with --compensate 0 it is
    the denoised signal.  int16 output follows the rule of the wav outputs with --peak."""
    neg = stream_context(ap, a.neg, "--neg")
    pos = None if _is_silent(a.pos) else stream_context(ap, a.pos, "--pos")
    eng = get_engine(VARIANT)
    [sid] = eng.stream_open(None if pos is None else [pos], [neg], [a.peak])

    def step(x, final):
        comp = eng.stream_step_post([sid], [x], a.compensate, final=[int(final)])["compensated"][0]
        return pcm_bytes(comp if a.float32 else _to_i16(comp, a.peak))
    try:
        stream_pipe(step, a.input, a.output, a.chunk_ms)
    finally:
        eng.stream_close([sid])


def main(argv=None):
    ap = argparse.ArgumentParser(prog="nhans_denoiser", description="N-HANS denoiser / selective noise suppression (B200 engine)")
    ap.add_argument("--input", default=FLAGS.input)
    ap.add_argument("--neg", default=FLAGS.neg)
    ap.add_argument("--pos", default=FLAGS.pos)
    ap.add_argument("--output", default=FLAGS.output)
    ap.add_argument("--compensate", type=float, default=0.0)
    ap.add_argument("--ac", action="store_true")
    ap.add_argument("--float32", action="store_true", help="write float32 wavs like the reference instead of 16-bit PCM")
    add_stream_args(ap)
    a = ap.parse_args(argv)
    if a.stream:
        if a.ac:
            ap.error("--ac cannot be used with --stream: its factor is the whole clip's snr_est, which a live stream does not "
                     "know until it ends; use --compensate")
        check_stream_args(ap, a)
        stream_denoiser(ap, a)
        return 0
    FLAGS.input, FLAGS.neg, FLAGS.pos, FLAGS.output = a.input, a.neg, a.pos, a.output
    FLAGS.compensate, FLAGS.ac, FLAGS.float32 = a.compensate, a.ac, a.float32
    if os.path.isdir(a.input):
        mixed, poss, negs, outs = _pairs(a.input, a.pos, a.neg, a.output)
        if mixed:
            apply_snc_batch(mixed, poss, negs, outs)
    elif _is_silent(a.pos):
        apply_denoiser(a.input, a.neg, a.output)
    else:
        apply_snc(a.input, a.pos, a.neg, a.output)
    return 0


if __name__ == "__main__":
    sys.exit(main())
