"""Drop-in mirror of N_HANS___Source_Separation/apply.py on the B200 engine.

``apply_separator(mixedpath, cleanpath, noisepath, save_to)`` (SS/apply.py:288-397) with the flags
``--input --pos(target speaker) --neg(interference speaker) --output`` (SS/apply.py:28-34), folder mode
(README.md:59-66) and ``main()`` (setup.py:48).  The reference feeds ``noisecontextph`` from --neg and
``cleancontextph`` from --pos (SS/apply.py:374-385); the engine calls them ctx_a / ctx_b.  It writes the
separated wav and '<...>mixed_processed.wav' (SS/apply.py:395-397)."""
from __future__ import annotations

import argparse
import os
import sys

import numpy as np

from .. import weights as W
from ..session import get_engine
from ..wavio import FS, is_pcm16, read_wav, write_wav
from ..selective_noise.apply import (_emit, _fit_noise, _norm64, _seq_sum, _sibling, add_stream_args, check_stream_args,
                                     pcm_bytes, stream_context, stream_pipe)

Noise_Win = 200
Mix_Win = 35
VARIANT = W.SEPARATOR


class _Flags:        # SS/apply.py:28-34
    input = "./audio_examples/mixed.wav"
    neg = "./audio_examples/noise_speaker.wav"
    pos = "./audio_examples/target_speaker.wav"
    output = "./audio_examples/denoised.wav"
    Fs = FS
    float32 = False


FLAGS = _Flags()


def handle_signals(mixedpath, cleanpath, noisepath):
    """SS/apply.py:111-136."""
    eng = get_engine(VARIANT)
    mixed = eng.normalise([read_wav(mixedpath)], trim=True)[0]
    clean = eng.normalise([read_wav(cleanpath)], trim=False)[0]
    noise = eng.normalise([read_wav(noisepath)], trim=False)[0]
    return clean, noise, mixed


def domixing(cleansamples, noisesamples, snr):
    """SS/apply.py:55-80 -> (mixed, K)."""
    sig = np.asarray(cleansamples, np.float32)
    nse = _fit_noise(np.asarray(noisesamples, np.float32), len(sig))
    psignal = _seq_sum(abs(sig) * abs(sig)) / sig.shape[0]
    pnoise = _seq_sum(abs(nse) * abs(nse)) / nse.shape[0]
    K = float(np.sqrt(1.0 if pnoise == 0 else (psignal / pnoise) * pow(10, -snr / 10.0)))
    mixed = sig + np.float32(K) * nse
    return mixed / np.float32(float(max(abs(mixed))) + 0.000001), K


def combine_signals(cleanpath, noisepath):
    """SS/apply.py:83-108 -> (clean, noise * K, mixed, snr).  The reference slices ``clean[:-rem]`` even when
    rem == 0 (which would empty the signal); a whole number of frames is kept as is here."""
    clean = _norm64(read_wav(cleanpath))
    noise = _norm64(read_wav(noisepath))
    rem = (len(clean) - 400) % 160
    if rem != 0:
        clean = clean[:-rem]
    snr = 0
    mixed, K = domixing(clean, noise, snr)
    return clean, noise * np.float32(K), mixed, np.array(snr, np.int32)


def apply_demo(cleanpath, noisepath, save_to):
    """SS/apply.py:179-285: on-the-fly 0 dB mixture of two speakers; contexts = first 200 frames of the clean
    (target) and the scaled interfering speaker; frames [200:] are separated.  Writes ``save_to`` and
    ``save_to[:-15] + 'mixed_demo.wav'``."""
    clean, noise_k, mixed, _ = combine_signals(cleanpath, noisepath)
    eng = get_engine(VARIANT)
    y, ymix = eng.enhance_demo(mixed, noise_k, clean, start=Noise_Win)      # ctx_a = interference, ctx_b = target
    write_wav(save_to, y)
    write_wav(save_to[:-15] + "mixed_demo.wav", ymix)
    return y, ymix


def recover_samples_from_spectrum(logspectrum_stft, spectrum_phase, save_to):
    """SS/apply.py:158-171."""
    eng = get_engine(VARIANT)
    lm = np.ascontiguousarray(logspectrum_stft, np.float32)
    samples, _ = eng.istft(lm, spectrum_phase, np.array([0, lm.shape[0]], np.int64))
    if save_to:
        write_wav(save_to, samples)
    return samples


def apply_separator_batch(mixedpaths, cleanpaths, noisepaths, save_tos, out_format=None):
    as_f32 = (FLAGS.float32 if out_format is None else out_format == "float32")
    eng = get_engine(VARIANT)
    mixes = [read_wav(p) for p in mixedpaths]
    cleans = [read_wav(p) for p in cleanpaths]
    noises = [read_wav(p) for p in noisepaths]
    U = len(mixes)
    pcm = [u for u in range(U) if is_pcm16(mixes[u]) and is_pcm16(cleans[u]) and is_pcm16(noises[u])]
    out = [None] * U
    if pcm:
        res = eng.enhance([mixes[u] for u in pcm], [noises[u] for u in pcm], [cleans[u] for u in pcm],
                          want_f32=True, want_i16=False, want_mixproc=True)                       # ctx_a = --neg, ctx_b = --pos
        for j, u in enumerate(pcm):
            out[u] = (res["f32"][j], res["mixed_processed"][j], float(max(abs(mixes[u]))) if len(mixes[u]) else 0.0)
    for u in range(U):
        if out[u] is None:                                         # a stereo file in the set: float entry points
            r = eng.enhance_float(mixes[u], noises[u], cleans[u])
            out[u] = (r["f32"], r["mixed_processed"], r["peak"])
    for u, save_to in enumerate(save_tos):
        den, mixed, peak = out[u]
        _emit(save_to, den, peak, as_f32)
        _emit(_sibling(save_to, "mixed_processed.wav"), mixed, peak, as_f32)


def apply_separator(mixedpath, cleanpath, noisepath, save_to):
    """SS/apply.py:288-397: extract the speaker of ``cleanpath`` (--pos), suppress the one of ``noisepath`` (--neg)."""
    apply_separator_batch([mixedpath], [cleanpath], [noisepath], [save_to])


def stream_separator(ap, a):
    """--stream: the separated signal of one live stream (int16 scaled by --peak, or float32)."""
    noise = stream_context(ap, a.neg, "--neg")
    clean = stream_context(ap, a.pos, "--pos")
    eng = get_engine(VARIANT)
    [sid] = eng.stream_open([noise], [clean], [a.peak])                     # ctx_a = --neg, ctx_b = --pos

    def step(x, final):
        r = eng.stream_step([sid], [x], final=[int(final)], want_f32=a.float32, want_i16=not a.float32)
        return pcm_bytes(r["f32"][0] if a.float32 else r["i16"][0])
    try:
        stream_pipe(step, a.input, a.output, a.chunk_ms)
    finally:
        eng.stream_close([sid])


def main(argv=None):
    ap = argparse.ArgumentParser(prog="nhans_separator", description="N-HANS speech separator (B200 engine)")
    ap.add_argument("--input", default=FLAGS.input)
    ap.add_argument("--neg", default=FLAGS.neg)
    ap.add_argument("--pos", default=FLAGS.pos)
    ap.add_argument("--output", default=FLAGS.output)
    ap.add_argument("--float32", action="store_true")
    add_stream_args(ap)
    a = ap.parse_args(argv)
    if a.stream:
        check_stream_args(ap, a)
        stream_separator(ap, a)
        return 0
    FLAGS.input, FLAGS.neg, FLAGS.pos, FLAGS.output, FLAGS.float32 = a.input, a.neg, a.pos, a.output, a.float32
    if os.path.isdir(a.input):
        names = sorted(f for f in os.listdir(a.input) if f.lower().endswith(".wav"))
        os.makedirs(a.output, exist_ok=True)
        names = [n for n in names if os.path.exists(os.path.join(a.pos, n)) and os.path.exists(os.path.join(a.neg, n))]
        if names:
            apply_separator_batch([os.path.join(a.input, n) for n in names], [os.path.join(a.pos, n) for n in names],
                                  [os.path.join(a.neg, n) for n in names],
                                  [os.path.join(a.output, n[:-4] + "_denoised.wav") for n in names])
    else:
        apply_separator(a.input, a.pos, a.neg, a.output)
    return 0


if __name__ == "__main__":
    sys.exit(main())
