"""End-to-end apply path through nhans_enhance_batch: SNR >= 40 dB against the oracle's apply_snc /
apply_separator restatement, golden vectors, batch invariance, error behaviour, CLI file surface."""
import os

import numpy as np
import pytest

from nhans_b200 import synth, weights as W
from nhans_b200.engine import Engine, NhansError
from oracle import nhans_oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
SNR_MIN_DB = 40.0


def _snr(ref, got):
    ref = ref.astype(np.float64)
    err = got.astype(np.float64) - ref
    return 10 * np.log10(np.sum(ref ** 2) / (np.sum(err ** 2) + 1e-30))


def test_denoiser_snr_vs_oracle(engine_sn, oracle_sn):
    mixes = [synth.mixture(1.0, 0), synth.mixture(0.6, 1), synth.mixture(0.35, 2)]      # ragged batch
    negs = [synth.noise_clip(u) for u in range(3)]
    res = engine_sn.enhance(mixes, None, negs, want_mixproc=True)
    for u in range(3):
        r = O.apply_arrays(oracle_sn, mixes[u], synth.silence(), negs[u], return_all=True)
        assert len(res["f32"][u]) == len(r["samples"])
        assert _snr(r["samples"], res["f32"][u]) >= SNR_MIN_DB
        assert np.abs(res["mixed_processed"][u] - r["mixed_processed"]).max() < 1e-5
        i16 = O.to_int16(r["samples"], r["peak"]).astype(np.int32)
        assert np.abs(res["i16"][u].astype(np.int32) - i16).max() <= max(2, int(3e-3 * np.abs(i16).max()))


def test_selective_noise_pos_and_neg(engine_sn, oracle_sn):
    mix, pos, neg = synth.mixture(0.5, 4), synth.noise_clip(4, "pos"), synth.noise_clip(4, "neg")
    res = engine_sn.enhance([mix], [pos], [neg])
    ref = O.apply_arrays(oracle_sn, mix, pos, neg)
    assert _snr(ref, res["f32"][0]) >= SNR_MIN_DB


def test_separator_snr_vs_oracle(engine_ss, oracle_ss):
    mix = synth.mixture(0.5, 6)
    tgt, itf = synth.speaker_clip(6, "target"), synth.speaker_clip(6, "interference")
    res = engine_ss.enhance([mix], [itf], [tgt])                     # ctx_a = --neg (interference), ctx_b = --pos (target)
    ref = O.apply_arrays(oracle_ss, mix, itf, tgt)
    assert _snr(ref, res["f32"][0]) >= SNR_MIN_DB
    with pytest.raises(NhansError):                                  # the separator has no Silent default
        engine_ss.enhance([mix], None, [tgt])


@pytest.mark.parametrize("tag", ["sn", "ss"])
def test_golden_vectors(tag, engine_sn, engine_ss):
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLD, "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    g = np.load(os.path.join(GOLD, "golden_%s.npz" % tag))
    eng = engine_sn if tag == "sn" else engine_ss
    mix, a, b = mg.inputs(tag)
    lm, ph, fo, _ = eng.stft([mix])
    assert np.abs(lm - g["logmag"]).max() < 1e-3
    res = eng.enhance([mix], None if tag == "sn" else [a], [b], want_mixproc=True)
    assert _snr(g["samples"], res["f32"][0]) >= SNR_MIN_DB
    assert np.abs(res["mixed_processed"][0] - g["mixed_processed"]).max() < 1e-5


def test_batch_invariance_and_chunking(engine_sn):
    """An utterance's output does not depend on its position in the batch or on the pass boundaries."""
    mixes = [synth.mixture(0.3 + 0.05 * (u % 5), u) for u in range(12)]       # ~470 windows, capacity 256 -> 2 passes
    negs = [synth.noise_clip(u % 3) for u in range(12)]
    res = engine_sn.enhance(mixes, None, negs)
    for u in (0, 5, 11):
        solo = engine_sn.enhance([mixes[u]], None, [negs[u]])
        assert np.array_equal(solo["i16"][0], res["i16"][u])
        assert np.array_equal(solo["f32"][0], res["f32"][u])


def test_zero_last_dense_identity(weights_sn):
    """SURVEY.md §4 (iii): with last_dense == 0 the denoised wav equals mixed_processed.wav exactly."""
    w = dict(weights_sn)
    w["last_dense/w"] = np.zeros_like(w["last_dense/w"])
    w["last_dense/b"] = np.zeros_like(w["last_dense/b"])
    eng = Engine(0, 0, win_capacity=64, row_capacity=1)
    eng.load_weights(w)
    res = eng.enhance([synth.mixture(0.4, 8)], None, [synth.noise_clip(8)], want_mixproc=True)
    assert np.array_equal(res["f32"][0], res["mixed_processed"][0])
    eng.close()


def test_error_behaviour(engine_sn):
    with pytest.raises(NhansError) as ei:                             # 1 s context: < 200 frames (SURVEY F9)
        engine_sn.enhance([synth.mixture(0.3, 0)], None, [synth.noise_clip(0, seconds=1.0)])
    assert ei.value.code == -4
    res = engine_sn.enhance([synth.mixture(0.3, 0)[:300], synth.mixture(0.3, 1)], None, [synth.noise_clip(0), synth.noise_clip(1)])
    assert len(res["f32"][0]) == 0 and len(res["f32"][1]) == O.trim_len(4800)     # < 400 samples -> no frames, empty output
    eng = Engine(0, 0, win_capacity=8, row_capacity=1)
    with pytest.raises(NhansError):                                   # weights not loaded
        eng.enhance([synth.mixture(0.3, 0)], None, [synth.noise_clip(0)])
    with pytest.raises(NhansError):
        eng.load_weights({"last_dense/w": np.zeros((3, 3), np.float32)})
    eng.close()


def test_cli_file_surface(tmp_path, monkeypatch):
    """nhans_denoiser / nhans_separator: 16 kHz 16-bit PCM in and out, the four SN outputs, folder mode."""
    from nhans_b200 import session
    from nhans_b200.selective_noise import apply as sn_apply
    from nhans_b200.source_separation import apply as ss_apply
    from nhans_b200.wavio import read_wav, write_wav
    monkeypatch.setenv("NHANS_WIN_CAPACITY", "128")
    monkeypatch.setenv("NHANS_ROW_CAPACITY", "2")
    monkeypatch.setenv("NHANS_MODEL_DIR", str(tmp_path / "no_model"))
    monkeypatch.setenv("NHANS_ALLOW_RANDOM_INIT", "1")            # no checkpoint on the test box: seeded random init
    session.close_all()
    d = tmp_path
    write_wav(str(d / "mixed.wav"), synth.mixture(0.5, 0))
    write_wav(str(d / "noise.wav"), synth.noise_clip(0))
    write_wav(str(d / "pos.wav"), synth.noise_clip(0, "pos"))
    out = str(d / "out_denoised.wav")
    assert sn_apply.main(["--input", str(d / "mixed.wav"), "--neg", str(d / "noise.wav"), "--output", out]) == 0
    for name in ("out_denoised.wav", "out_mixed_processed.wav", "out_removed.wav", "out_compensated.wav"):
        y = read_wav(str(d / name))                                   # asserts 16 kHz int16
        assert len(y) == O.trim_len(8000)
    a = read_wav(out)
    sn_apply.apply_snc(str(d / "mixed.wav"), str(d / "pos.wav"), str(d / "noise.wav"), str(d / "snc_denoised.wav"))
    assert not np.array_equal(read_wav(str(d / "snc_denoised.wav")), a)          # the --pos context matters
    # folder mode (README.md:59-66)
    for sub in ("in", "neg"):
        os.makedirs(str(d / sub))
    for n in ("a.wav", "b.wav"):
        write_wav(str(d / "in" / n), synth.mixture(0.3, 3))
        write_wav(str(d / "neg" / n), synth.noise_clip(3))
    assert sn_apply.main(["--input", str(d / "in"), "--neg", str(d / "neg"), "--output", str(d / "outdir")]) == 0
    assert sorted(f for f in os.listdir(str(d / "outdir")) if f.endswith("_denoised.wav")) == ["a_denoised.wav", "b_denoised.wav"]
    write_wav(str(d / "tgt.wav"), synth.speaker_clip(1, "target"))
    write_wav(str(d / "itf.wav"), synth.speaker_clip(1, "interference"))
    assert ss_apply.main(["--input", str(d / "mixed.wav"), "--pos", str(d / "tgt.wav"), "--neg", str(d / "itf.wav"),
                          "--output", str(d / "sep_denoised.wav"), "--float32"]) == 0
    from scipy.io.wavfile import read
    rate, y = read(str(d / "sep_denoised.wav"))
    assert rate == 16000 and y.dtype == np.float32                    # the reference's own output format
    session.close_all()


def test_postmix_outputs_vs_oracle(engine_sn, oracle_sn):
    """SN/apply.py:456-470 on the GPU (fused dual iSTFT + energy sums): removed, snr_est, compensated."""
    mixes = [synth.mixture(0.6, 2), synth.mixture(0.4, 3)]
    negs = [synth.noise_clip(2), synth.noise_clip(3)]
    res = engine_sn.enhance(mixes, None, negs)
    for ac, comp in ((False, 0.3), (True, 0.0)):
        post = engine_sn.postmix(res["out_offs"], compensate=comp, ac=ac)
        for u in range(2):
            r = O.apply_arrays(oracle_sn, mixes[u], synth.silence(), negs[u], return_all=True)
            removed, snr_est, compensated = O.post_mix(r["samples"], r["mixed_processed"], comp, ac)
            assert np.abs(post["mixed_processed"][u] - r["mixed_processed"]).max() < 1e-5
            assert _snr(removed, post["removed"][u]) >= 30.0          # removed is a small difference of two signals
            assert abs(post["snr_est"][u] - snr_est) <= 5e-3 * abs(snr_est)
            assert _snr(compensated, post["compensated"][u]) >= SNR_MIN_DB
            assert np.abs(post["removed"][u] - (post["mixed_processed"][u] - res["f32"][u])).max() < 1e-5


def test_many_tiny_utterances(engine_sn, oracle_sn):
    """300 utterances of 2-4 frames: a full pass would need more virtual frames than the per-frame convolution table
    holds, so the batch is split into smaller passes that fit it; every window is mostly zero padding.  An
    utterance's result does not depend on which others share its pass."""
    rng = np.random.default_rng(5)
    base = synth.mixture(1.0, 9)
    mixes = [base[o:o + int(rng.integers(560, 1040))] for o in rng.integers(0, 12000, 300)]
    neg = synth.noise_clip(9)
    res = engine_sn.enhance(mixes, None, [neg] * 300)
    for u in (0, 57, 299):
        ref = O.apply_arrays(oracle_sn, mixes[u], synth.silence(), neg)
        assert len(res["f32"][u]) == len(ref) == O.trim_len(len(mixes[u]))
        assert _snr(ref, res["f32"][u]) >= SNR_MIN_DB
    solo = engine_sn.enhance([mixes[123]], None, [neg])
    assert _snr(solo["f32"][0], res["f32"][123]) >= 60.0
    assert np.array_equal(solo["f32"][0], res["f32"][123])


def test_multigpu_runtime_scatter_gather(engine_sn, weights_sn):
    """runtime.MultiGpu: one engine per device, one host thread each, ragged batch dealt by load, results gathered
    back in input order.  Two contexts on device 0 stand in for two GPUs (the data path has no collective)."""
    from nhans_b200.runtime import MultiGpu
    mixes = [synth.mixture(0.25 + 0.1 * (u % 4), 70 + u) for u in range(9)]
    negs = [synth.noise_clip(70 + u % 2) for u in range(9)]
    mg = MultiGpu([0, 0], W.SELECTIVE_NOISE, weights_sn, win_capacity=128, row_capacity=2)
    try:
        got = mg.enhance(mixes, None, negs)
    finally:
        mg.close()
    ref = engine_sn.enhance(mixes, None, negs)
    assert len(got["i16"]) == 9
    for u in range(9):
        assert np.array_equal(got["i16"][u], ref["i16"][u])
        assert np.array_equal(got["f32"][u], ref["f32"][u])


def test_pipelined_batches_match_sequential(engine_sn):
    """Two batches in flight (double-buffered staging + the library's copy streams): submit A, submit B, collect A
    while B still runs, collect B - bit-identical to processing them one after the other; a third submit before a
    collect is refused."""
    A = ([synth.mixture(0.5, 80), synth.mixture(0.3, 81)], None, [synth.noise_clip(80), synth.noise_clip(81)])
    B = ([synth.mixture(0.45, 82)], None, [synth.noise_clip(82)])
    ra, rb = engine_sn.enhance(*A), engine_sn.enhance(*B)
    ta = engine_sn.submit(*A)
    tb = engine_sn.submit(*B)
    with pytest.raises(NhansError):
        engine_sn.submit(*B)
    ga = engine_sn.collect(ta, newer_in_flight=True)
    gb = engine_sn.collect(tb)
    for got, want in ((ga, ra), (gb, rb)):
        for u in range(len(want["i16"])):
            assert np.array_equal(got["i16"][u], want["i16"][u]) and np.array_equal(got["f32"][u], want["f32"][u])
    # many alternating batches: staging sets and events are reused correctly
    prev = None
    for k in range(6):
        cur = engine_sn.submit(*(A if k % 2 == 0 else B))
        if prev is not None:
            g = engine_sn.collect(prev[0], newer_in_flight=True)
            want = ra if prev[1] % 2 == 0 else rb
            assert all(np.array_equal(g["i16"][u], want["i16"][u]) for u in range(len(want["i16"])))
        prev = (cur, k)
    g = engine_sn.collect(prev[0])
    assert np.array_equal(g["i16"][0], rb["i16"][0])
