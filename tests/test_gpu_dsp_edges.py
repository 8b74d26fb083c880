"""The signal ends of the engine (dsp.cu: stft_kernel, istft_kernel, istft_post_kernel, istft_stream_kernel,
compensate_kernel) against the float64 references of tests/dsp64.py, elementwise, at the kernels' block edges:
- forward: 4 frames per warp, 16 per CTA, and the int16 span staged by a bulk copy from the 16-byte boundary below its
  first sample (shift 0-7 samples);
- inverse: 26 output hops per CTA, T + 2 hops per clip, and the 3-frame gather that takes the third frame only for
  the first 80 samples of a hop;
- int16 output at both saturation ends, in the batch path and in live streams opened at peak 32767;
- post-mix sums over 1-5 inverse CTAs per clip, and clips without frames.
The fused-path checks read the spectra the kernels left in HBM, so the network is out of the loop and every bound is a
bound on the transform kernels alone.  Each check prints its measured maximum next to its bound."""
import numpy as np
import pytest

import dsp64 as R
from nhans_b200 import synth, weights as W
from nhans_b200.engine import Engine
from oracle import nhans_oracle as O

pytestmark = pytest.mark.gpu

# Bounds, each <= 4x the maximum measured on a B200 (DESIGN.md parity table).  Spectra: complex error of
# (exp(logmag) - 1e-5) * phasor per frame, relative to the frame's largest |X| (floored at 1e-4: below that the 1e-5 of
# log(|X| + 1e-5) leaves no resolution); log-magnitude on bins >= 1e-3 of the frame max; waveforms relative to the
# clip's largest value of |y| or of the unwindowed inverse FFT of its frames (a frame of zero samples has the spectrum
# 1e-5 with phasor (1, 0), whose inverse FFT is an impulse at the frame's first sample, where the window is 0: the
# output is 0 in exact arithmetic, and the kernel's fp32 rounding is relative to the impulse).
EPS_SPEC = 2.5e-6
EPS_LOGMAG = 2e-4
EPS_UNIT = 6e-7
EPS_WAVE = 2.4e-6
EPS_SNR = 2e-7
FRAME_FLOOR = 1e-4

KINDS = ("mix", "square", "impulse", "const", "alt", "zeros")


def _report(name, measured, bound):
    print("%-34s max %.3g  (bound %.3g)" % (name, measured, bound))
    assert measured <= bound, "%s: %.3g > %.3g" % (name, measured, bound)


def _signal(kind, n, seed):
    i = np.arange(n)
    if kind == "mix":
        return synth.mixture(0.7, seed % 11)[:n].copy()
    if kind == "square":                                  # full scale, with the -32768 that abs() wraps
        return np.where((i // 37) % 2 == 0, 32767, -32768).astype(np.int16)
    if kind == "impulse":
        x = np.zeros(n, np.int16)
        x[(seed * 97) % n] = 1234
        return x
    if kind == "const":
        return np.full(n, 12345, np.int16)
    if kind == "alt":                                     # Nyquist
        return np.where(i % 2 == 0, 23456, -23456).astype(np.int16)
    return np.zeros(n, np.int16)


def _edge_clips():
    """T = 1..40, 63, 64, 65 frames, each with tails of 0, 1, 79 and 159 samples past the last frame, cycling through
    KINDS.  Before each one a clip of < 400 samples (no frame) moves the next clip's first sample to the residue
    k mod 8 of a 16-byte boundary, so the framed clips cover every shift of the bulk copy."""
    clips, off, k = [], 0, 0
    for T in list(range(1, 41)) + [63, 64, 65]:
        for r in (0, 1, 79, 159):
            fill = (k % 8 - off) % 8 or 8
            fill += 160 * (k % 3)
            clips.append(_signal("mix", fill, k))
            n = 400 + 160 * (T - 1) + r
            clips.append(_signal(KINDS[k % len(KINDS)], n, k))
            off += fill + n
            k += 1
    return clips


def _starts(clips):
    return np.cumsum([0] + [len(c) for c in clips])[:-1]


def _spec_errors(logmag, phasor, X):
    """-> (complex error per frame / max(frame max, FRAME_FLOOR), log-magnitude error on bins >= 1e-3 of the frame
    max), maxima over the frames of one clip."""
    mag = np.exp(logmag.astype(np.float64)) - R.LOG_EPS
    fmax = np.abs(X).max(axis=1)
    cplx = (np.abs(mag * phasor - X).max(axis=1) / np.maximum(fmax, FRAME_FLOOR)).max()
    big = np.abs(X) >= 1e-3 * fmax[:, None]
    big &= fmax[:, None] >= FRAME_FLOOR
    lm_err = np.abs(logmag.astype(np.float64) - np.log(np.abs(X) + R.LOG_EPS))[big]
    return cplx, (lm_err.max() if lm_err.size else 0.0)


def _wave_error(got, logmag, phasor):
    """Inverse STFT of exp(logmag) * phasor: error of `got` against istft64, relative to the clip's scale (above)."""
    mag = np.exp(logmag.astype(np.float64))
    ref = R.istft64(mag, phasor)
    assert len(got) == len(ref)
    if not len(ref):
        return 0.0
    scale = max(np.abs(ref).max(), np.abs(np.fft.irfft(mag * phasor, n=R.WIN, axis=1)).max())
    return np.abs(got.astype(np.float64) - ref).max() / scale


def _phasor(ph):
    return ph[..., 0].astype(np.float64) + 1j * ph[..., 1].astype(np.float64)


def _check_fused_spectra(name, clips, fo, lm, ph, den, res):
    """Phasor spectra of the fused path against stft64, and both inverse transforms (denoised -> f32, input spectrum ->
    mixed_processed) against istft64 of the very spectra the kernels read; int16 follows the output rule."""
    e_c = e_l = e_u = e_d = e_m = 0.0
    for u, c in enumerate(clips):
        a, b = fo[u], fo[u + 1]
        X = R.stft64(R.normalise_i16(c))
        assert b - a == X.shape[0]
        if b == a:
            assert len(res["f32"][u]) == len(res["mixed_processed"][u]) == len(res["i16"][u]) == 0
            continue
        P = _phasor(ph[a:b])
        c_err, l_err = _spec_errors(lm[a:b], P, X)
        e_c, e_l = max(e_c, c_err), max(e_l, l_err)
        silent = ~np.abs(X).any(axis=1)                  # frames of zero samples: every bin takes the r2 = 0 branch
        assert np.all(ph[a:b][silent] == np.array([1.0, 0.0], np.float32))
        live = np.abs(X) ** 2 > 1e-29
        if live.any():
            e_u = max(e_u, np.abs(np.abs(P[live]) - 1).max())
        e_d = max(e_d, _wave_error(res["f32"][u], den[a:b], P))
        e_m = max(e_m, _wave_error(res["mixed_processed"][u], lm[a:b], P))
        assert np.array_equal(res["i16"][u], R.i16_rule(res["f32"][u], O.peak_of(c)))
    _report(name + ": stft phasor spectrum", e_c, EPS_SPEC)
    _report(name + ": stft log-magnitude", e_l, EPS_LOGMAG)
    _report(name + ": phasor |.| - 1", e_u, EPS_UNIT)
    _report(name + ": istft denoised", e_d, EPS_WAVE)
    _report(name + ": istft mixed_processed", e_m, EPS_WAVE)


@pytest.fixture(scope="module")
def boosted(weights_sn):
    """last_dense = 0 with bias log 2: the mask multiplies every magnitude by 2, so outputs are about twice the input
    and a full-scale clip saturates int16."""
    w = dict(weights_sn)
    w["last_dense/w"] = np.zeros_like(w["last_dense/w"])
    w["last_dense/b"] = np.full_like(w["last_dense/b"], np.log(2.0))
    e = Engine(0, W.SELECTIVE_NOISE, win_capacity=256, row_capacity=4)
    e.load_weights(w)
    yield e
    e.close()


def test_edge_clips_cover_every_bulk_copy_shift():
    clips = _edge_clips()
    framed = [int(s) % 8 for s, c in zip(_starts(clips), clips) if len(c) >= 400]
    assert sorted(set(framed)) == list(range(8))
    assert sum(len(c) < 400 for c in clips) == len(framed) == 43 * 4


def test_stft_entries_at_block_edges(engine_sn):
    """nhans_stft (int16, angles) and nhans_stft_f32 (float, angles) on one batch of every block edge."""
    clips = _edge_clips()
    lm, ph, fo, peak = engine_sn.stft(clips)
    assert fo.tolist() == np.cumsum([0] + [R.n_frames(len(c)) for c in clips]).tolist()
    xs = [O.normalise(c) for c in clips]
    lm2, ph2, fo2 = engine_sn.stft_f32(xs)
    assert np.array_equal(fo2, fo)
    errs = {}
    for u, (c, x) in enumerate(zip(clips, xs)):
        assert int(peak[u]) == int(O.peak_of(c))
        a, b = fo[u], fo[u + 1]
        if a == b:
            continue
        X = R.stft64(x)
        for key, l, p in (("nhans_stft", lm, ph), ("nhans_stft_f32", lm2, ph2)):
            c_err, l_err = _spec_errors(l[a:b], np.exp(1j * p[a:b].astype(np.float64)), X)
            e = errs.setdefault(key, [0.0, 0.0])
            e[0], e[1] = max(e[0], c_err), max(e[1], l_err)
    for key, (c_err, l_err) in errs.items():
        _report(key + ": complex spectrum", c_err, EPS_SPEC)
        _report(key + ": log-magnitude", l_err, EPS_LOGMAG)


def test_fused_path_at_block_edges(engine_sn):
    """The same batch through enhance: the phasor STFT and both phasor inverse transforms, from the engine's own
    spectra, plus the int16 rule on every sample."""
    clips = _edge_clips()
    ctx = [synth.noise_clip(u % 5) for u in range(len(clips))]
    res = engine_sn.enhance(clips, None, ctx, want_mixproc=True)
    fo = np.cumsum([0] + [R.n_frames(len(c)) for c in clips])
    lm, ph, den = engine_sn.read_batch_spectra(int(fo[-1]))
    _check_fused_spectra("edges", clips, fo, lm, ph, den, res)


def test_fused_path_production_batch():
    """A benchmark-sized batch (256 x 4 s, 101888 frames) through one fused call of a default-capacity engine: every
    frame's spectrum and every output sample."""
    eng = Engine(0, W.SELECTIVE_NOISE)
    try:
        eng.load_weights(W.seeded_init(W.SELECTIVE_NOISE, 0))
        base_m = [synth.mixture(4.0, u) for u in range(16)]
        base_n = [synth.noise_clip(u) for u in range(16)]
        order = [(7 * u + 3) % 16 for u in range(256)]
        clips = [base_m[i] for i in order]
        res = eng.enhance(clips, None, [base_n[i] for i in order], want_mixproc=True)
        fo = np.cumsum([0] + [R.n_frames(len(c)) for c in clips])
        assert fo[-1] == 256 * 398
        lm, ph, den = eng.read_batch_spectra(int(fo[-1]))
    finally:
        eng.close()
    _check_fused_spectra("256 x 4 s", clips, fo, lm, ph, den, res)


def test_istft_angles_at_hop_block_edges(engine_sn):
    """nhans_istft (angles) for T = 1..60, 76, 77 (T + 2 = 26, 27, 52, 53, 78, 79 hops sit on CTA edges), clips without
    frames in between, random spectra and spectra of clips that reach 1.5x full scale; int16 at peaks 0, 1, 1000 and
    32767 follows the output rule bit for bit, saturating at both ends."""
    rng = np.random.default_rng(3)
    lms, phs, T_list, peaks = [], [], [], []
    for j, T in enumerate(list(range(1, 61)) + [76, 77]):
        if j % 5 == 0:
            T_list.append(0)
            peaks.append(32767)
        if j % 2:
            lm = rng.normal(-1.0, 1.5, (T, 201)).astype(np.float32)
            ph = rng.uniform(-np.pi, np.pi, (T, 201)).astype(np.float32)
        else:
            x = O.normalise(synth.mixture(1.0, j))[:400 + 160 * (T - 1)] * np.float32(1.5)
            X = R.stft64(x)
            lm, ph = np.log(np.abs(X) + R.LOG_EPS).astype(np.float32), np.angle(X).astype(np.float32)
        lms.append(lm)
        phs.append(ph)
        T_list.append(T)
        peaks.append((0, 1, 1000, 32767)[j % 4])
    lm, ph = np.concatenate(lms), np.concatenate(phs)
    fo = np.cumsum([0] + T_list)
    y, i16, oo = engine_sn.istft(lm, ph, fo, peak=np.array(peaks, np.int32), want_i16=True)
    err, sat = 0.0, set()
    for u in range(len(T_list)):
        a, b = fo[u], fo[u + 1]
        got, q = y[oo[u]:oo[u + 1]], i16[oo[u]:oo[u + 1]]
        err = max(err, _wave_error(got, lm[a:b], np.exp(1j * ph[a:b].astype(np.float64))))
        assert np.array_equal(q, R.i16_rule(got, peaks[u]))
        if peaks[u] == 32767:
            sat |= set(np.intersect1d(q, [-32768, 32767]).tolist())
    _report("nhans_istft angles", err, EPS_WAVE)
    assert sat == {-32768, 32767}


def test_i16_saturation_fused_batch(boosted):
    """Boosted mask: outputs about twice the input, so full-scale clips saturate; int16 equals the output rule applied
    to the float32 output of the same call, sample for sample."""
    clips = [synth.mixture(0.9, 30), synth.mixture(0.45, 31)[:399], synth.mixture(0.6, 32)]
    loud = clips[2].copy()
    loud[::97] = -32768
    clips.append(loud)
    res = boosted.enhance(clips, None, [synth.noise_clip(u) for u in range(4)])
    sat = set()
    for u, c in enumerate(clips):
        assert np.array_equal(res["i16"][u], R.i16_rule(res["f32"][u], O.peak_of(c)))
        sat |= set(np.intersect1d(res["i16"][u], [-32768, 32767]).tolist())
    assert sat == {-32768, 32767}


def _live_oracle(net, pcm, ctx_b):
    """apply_snc with the mixture scaled by the live peak, x / (32767 + 1e-6), instead of its own max|x|."""
    mix = (np.asarray(pcm, np.float64) / (32767 + 0.000001)).astype(np.float32)
    lm, ph = O.logmag_phase(mix[:O.trim_len(len(mix))])
    ca = O.context_of(O.logmag_phase(O.normalise(synth.silence()))[0])
    cb = O.context_of(O.logmag_phase(O.normalise(ctx_b))[0])
    import torch
    with torch.no_grad():
        ea, eb = net.tower(O._t(ca, torch.float32)[None]), net.tower(O._t(cb, torch.float32)[None])
        win = O._t(O.strided_crop(lm, O.MIX_WIN, 1), torch.float32)
        den = torch.cat([net.mask_net(win[i:i + 100], ea.expand(len(win[i:i + 100]), -1), eb.expand(len(win[i:i + 100]), -1))
                         for i in range(0, len(win), 100)]).numpy()
    return O.istft(den, ph)


def _stream_live(eng, pcm, ctx_b, chunk):
    [sid] = eng.stream_open(None, [ctx_b], [32767])
    steps = []
    for s in range(0, len(pcm), chunk):
        r = eng.stream_step([sid], [pcm[s:s + chunk]], final=[int(s + chunk >= len(pcm))])
        steps.append((r["i16"][0], r["f32"][0]))
    eng.stream_close([sid])
    return steps


def test_live_peak_streams(boosted, engine_sn, oracle_sn):
    """Streams opened at the live peak 32767 (INTEGRATION.md): with the boosted mask every step's int16 is the output
    rule of that step's float32 and saturates at both ends; with the seeded weights the stream matches the oracle
    with its normalisation replaced by x / (32767 + 1e-6)."""
    pcm = np.clip(synth.mixture(1.5, 33).astype(np.int32) * 2, -32768, 32767).astype(np.int16)
    neg = synth.noise_clip(33)
    sat = set()
    for q, y in _stream_live(boosted, pcm, neg, 1600):
        assert np.array_equal(q, R.i16_rule(y, 32767))
        sat |= set(np.intersect1d(q, [-32768, 32767]).tolist())
    assert sat == {-32768, 32767}
    y = np.concatenate([y for _, y in _stream_live(engine_sn, pcm, neg, 1600)])
    ref = _live_oracle(oracle_sn, pcm, neg).astype(np.float64)
    assert len(y) == len(ref) == O.trim_len(len(pcm))
    snr = 10 * np.log10(np.sum(ref ** 2) / (np.sum((y - ref) ** 2) + 1e-30))
    print("live stream vs oracle: %.1f dB" % snr)
    assert snr >= 40.0


def test_postmix_over_inverse_ctas(engine_sn):
    """Post-mix of clips with 1-5 inverse CTAs (26 hops each) and a clip without frames, from the engine's own
    outputs: removed = mixed_processed - f32 bit for bit, snr_est the float64 ratio of the sums, compensated within
    1 ulp of den + removed * factor (the kernel may fuse the multiply-add)."""
    Ts = [1, 2, 24, 25, 26, 0, 50, 51, 52, 76, 77, 78, 102, 103, 104, 128, 129, 130]
    base = synth.mixture(1.4, 40)
    clips = [base[37 * i:37 * i + 400 + 160 * (T - 1)] if T else base[:250] for i, T in enumerate(Ts)]
    res = engine_sn.enhance(clips, None, [synth.noise_clip(u % 3) for u in range(len(Ts))])
    fo = np.cumsum([0] + Ts)
    lm, ph, _ = engine_sn.read_batch_spectra(int(fo[-1]))
    e_m = e_s = 0.0
    for ac, comp in ((False, 0.3), (True, 0.0)):
        post = engine_sn.postmix(res["out_offs"], compensate=comp, ac=ac)
        for u, T in enumerate(Ts):
            den, mixed = res["f32"][u], post["mixed_processed"][u]
            if T:
                e_m = max(e_m, _wave_error(mixed, lm[fo[u]:fo[u + 1]], _phasor(ph[fo[u]:fo[u + 1]])))
            removed, snr, _, factor = R.postmix64(den, mixed, comp, ac)
            assert np.array_equal(post["removed"][u], removed)
            if T == 0:
                assert snr == np.inf and post["snr_est"][u] == np.inf and len(post["compensated"][u]) == 0
                continue
            e_s = max(e_s, abs(float(post["snr_est"][u]) - snr) / snr)
            # ac: the kernel's factor is float32(snr / 20) of its own sums, which snr_est reports rounded to float32
            f = np.float32(float(post["snr_est"][u]) / 20.0) if ac else factor
            exact = den.astype(np.float64) + removed.astype(np.float64) * np.float64(f)
            tol = np.spacing(np.abs(exact).astype(np.float32)).astype(np.float64)
            if ac:
                tol += np.abs(removed) * np.spacing(f)
            assert np.all(np.abs(post["compensated"][u].astype(np.float64) - exact) <= tol)
    _report("postmix mixed_processed", e_m, EPS_WAVE)
    _report("postmix snr_est (relative)", e_s, EPS_SNR)


def test_postmix_of_a_batch_without_frames(engine_sn):
    """A batch whose clips are all shorter than one frame: empty outputs and snr_est = +inf, whatever the batch before
    left in the engine."""
    res = engine_sn.enhance([synth.mixture(0.5, 41)], None, [synth.noise_clip(1)])
    assert np.isfinite(engine_sn.postmix(res["out_offs"])["snr_est"][0])
    res = engine_sn.enhance([synth.mixture(0.1, 42)[:399], synth.mixture(0.1, 43)[:5]], None,
                            [synth.noise_clip(2), synth.noise_clip(3)])
    for ac in (False, True):
        post = engine_sn.postmix(res["out_offs"], compensate=0.5, ac=ac)
        assert post["snr_est"].tolist() == [np.inf, np.inf]
        assert all(len(v) == 0 for k in ("mixed_processed", "removed", "compensated") for v in post[k])
