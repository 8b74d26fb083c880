"""Streaming enhancement (nhans_stream_open / step / close): for every chunking, a stream's concatenated output equals
the batch path's output for the whole clip bit for bit (int16 and float32, same peak and contexts), many streams share
network passes without changing each other's bits, the batch path is undisturbed, and argument errors leave the
context usable."""
import ctypes

import numpy as np
import pytest

from nhans_b200 import _lib, synth, weights as W
from nhans_b200.engine import Engine, NhansError

pytestmark = pytest.mark.gpu

RANDOM_SIZES = [0, 1, 159, 160, 161, 399, 400, 2960, 7919]
# < 400 samples, 20 frames, 40 frames (+ a partial hop), 4 s
LENGTHS = [300, 400 + 19 * 160, 400 + 39 * 160 + 77, 64000]


def _engine(variant, weights, cap):
    e = Engine(0, variant, win_capacity=cap, row_capacity=4)
    e.load_weights(weights)
    return e


@pytest.fixture(scope="module")
def sn(weights_sn):
    e = _engine(W.SELECTIVE_NOISE, weights_sn, 256)
    yield e
    e.close()


@pytest.fixture(scope="module")
def ss(weights_ss):
    e = _engine(W.SEPARATOR, weights_ss, 256)
    yield e
    e.close()


def _emit_len(before, after, final):
    e = ctypes.c_int64()
    assert _lib.load().nhans_stream_emit_len(before, after, int(final), ctypes.byref(e)) == 0
    return e.value


def _chunking(kind, n, rng):
    if kind == "one":
        return [n]
    if kind == "1600":
        return [1600] * (n // 1600) + ([n % 1600] if n % 1600 else [])
    sizes, left = [], n
    while left > 0:
        s = min(int(rng.choice(RANDOM_SIZES)), left)
        sizes.append(s)
        left -= s
    return sizes


def _peak(eng, mix):
    return int(eng.stft([mix])[3][0])


def _stream(eng, mix, ctx_a, ctx_b, sizes, empty_final=False):
    """Feed mix in chunks of `sizes` (the last one final unless empty_final) -> concatenated (i16, f32)."""
    [sid] = eng.stream_open(None if ctx_a is None else [ctx_a], [ctx_b], [_peak(eng, mix)])
    got16, got32, n = [], [], 0
    steps = [(s, False) for s in sizes[:-1]] + [(sizes[-1] if sizes else 0, not empty_final)]
    if empty_final:
        steps.append((0, True))
    for size, final in steps:
        r = eng.stream_step([sid], [mix[n:n + size]], final=[int(final)])
        assert len(r["i16"][0]) == len(r["f32"][0]) == _emit_len(n, n + size, final)
        n += size
        got16.append(r["i16"][0])
        got32.append(r["f32"][0])
    assert n == len(mix)
    eng.stream_close([sid])
    return np.concatenate(got16), np.concatenate(got32)


def _assert_equal(got, want):
    assert len(got[0]) == len(want["i16"][0])
    assert np.array_equal(got[0], want["i16"][0])
    assert np.array_equal(got[1], want["f32"][0])


@pytest.mark.parametrize("case", ["sn_silent", "sn_pos_neg", "ss"])
def test_stream_bit_identical_to_batch(case, sn, ss):
    rng = np.random.default_rng(1)
    eng = ss if case == "ss" else sn
    for li, length in enumerate(LENGTHS):
        mix = synth.mixture(4.2, 20 + li)[:length]
        if case == "sn_silent":
            ctx_a, ctx_b = None, synth.noise_clip(20 + li)
        elif case == "sn_pos_neg":
            ctx_a, ctx_b = synth.noise_clip(20 + li, "pos"), synth.noise_clip(20 + li, "neg")
        else:
            ctx_a, ctx_b = synth.speaker_clip(20 + li, "interference"), synth.speaker_clip(20 + li, "target")
        want = eng.enhance([mix], None if ctx_a is None else [ctx_a], [ctx_b])
        for kind in ("one", "1600", "random"):
            _assert_equal(_stream(eng, mix, ctx_a, ctx_b, _chunking(kind, len(mix), rng)), want)
        _assert_equal(_stream(eng, mix, ctx_a, ctx_b, _chunking("random", len(mix), rng), empty_final=True), want)


def test_many_streams_ragged_lifetimes(weights_sn, sn):
    """40 streams open and finish at different steps on an engine whose passes hold 64 windows, so passes split inside
    segments; each stream equals its batch result from an engine of another capacity."""
    rng = np.random.default_rng(2)
    eng = _engine(W.SELECTIVE_NOISE, weights_sn, 64)
    try:
        S = 40
        mixes = [synth.mixture(0.2 + 0.05 * (u % 9), 100 + u)[:int(rng.integers(300, 24000))] for u in range(S)]
        negs = [synth.noise_clip(100 + u % 4) for u in range(S)]
        want = sn.enhance(mixes, None, negs)
        opens = rng.integers(0, 12, S)
        ids, pos, out16, out32 = {}, [0] * S, [[] for _ in range(S)], [[] for _ in range(S)]
        for step in range(200):
            for u in [u for u in range(S) if opens[u] == step]:
                ids[u] = eng.stream_open(None, [negs[u]], [_peak(eng, mixes[u])])[0]
            live = [u for u in ids if ids[u] is not None and rng.random() < 0.8]
            if not live:
                if all(v is None for v in ids.values()) and len(ids) == S:
                    break
                continue
            chunks, finals = [], []
            for u in live:
                size = int(rng.choice([0, 160, 1600, 3331]))
                chunks.append(mixes[u][pos[u]:pos[u] + size])
                finals.append(int(pos[u] + size >= len(mixes[u]) and rng.random() < 0.5))
            r = eng.stream_step([ids[u] for u in live], chunks, final=finals)
            for k, u in enumerate(live):
                assert len(r["i16"][k]) == _emit_len(pos[u], pos[u] + len(chunks[k]), finals[k])
                pos[u] += len(chunks[k])
                out16[u].append(r["i16"][k])
                out32[u].append(r["f32"][k])
                if finals[k]:
                    eng.stream_close([ids[u]])
                    ids[u] = None
        assert len(ids) == S and all(v is None for v in ids.values())
        for u in range(S):
            assert np.array_equal(np.concatenate(out16[u]), want["i16"][u]), u
            assert np.array_equal(np.concatenate(out32[u]), want["f32"][u]), u
    finally:
        eng.close()


def test_reference_path_without_generated_operand(weights_sn, monkeypatch):
    """NHANS_NO_GEN=1: window_expand_kernel builds the first activation from the per-frame table, context frames included."""
    monkeypatch.setenv("NHANS_NO_GEN", "1")
    eng = _engine(W.SELECTIVE_NOISE, weights_sn, 128)
    try:
        rng = np.random.default_rng(3)
        for li, length in enumerate(LENGTHS[1:]):
            mix, neg = synth.mixture(4.2, 40 + li)[:length], synth.noise_clip(40 + li)
            want = eng.enhance([mix], None, [neg])
            _assert_equal(_stream(eng, mix, None, neg, _chunking("random", len(mix), rng)), want)
    finally:
        eng.close()


def test_stream_steps_leave_batch_results_alone(sn):
    A = ([synth.mixture(0.5, 60), synth.mixture(0.3, 61)], None, [synth.noise_clip(60), synth.noise_clip(61)])
    ref = sn.enhance(*A)
    post_ref = sn.postmix(ref["out_offs"], compensate=0.3)
    mix, neg = synth.mixture(1.0, 62), synth.noise_clip(62)
    [sid] = sn.stream_open(None, [neg], [32767])
    # a step while a submitted batch is in flight
    t = sn.submit(*A)
    sn.stream_step([sid], [mix[:8000]])
    got = sn.collect(t)
    for u in range(2):
        assert np.array_equal(got["i16"][u], ref["i16"][u]) and np.array_equal(got["f32"][u], ref["f32"][u])
    # a step between run and postmix / download
    from nhans_b200.engine import pack
    m, mo = pack(A[0])
    b, bo = pack(A[2])
    sn.upload(m, mo, None, None, b, bo)
    sn.run()
    sn.stream_step([sid], [mix[8000:]], final=[1])
    n = int(ref["out_offs"][-1])
    o16, o32 = np.zeros(n, np.int16), np.zeros(n, np.float32)
    sn.download(o16, o32)
    sn.sync()
    assert np.array_equal(o16, np.concatenate(ref["i16"])) and np.array_equal(o32, np.concatenate(ref["f32"]))
    post = sn.postmix(ref["out_offs"], compensate=0.3)
    for k in ("mixed_processed", "removed", "compensated"):
        for u in range(2):
            assert np.array_equal(post[k][u], post_ref[k][u]), k
    assert np.array_equal(post["snr_est"], post_ref["snr_est"])
    sn.stream_close([sid])


def test_stream_argument_errors_leave_the_context_usable(sn, weights_sn):
    mix, neg = synth.mixture(0.6, 70), synth.noise_clip(70)
    want = sn.enhance([mix], None, [neg])

    def code(fn, *args, **kw):
        with pytest.raises(NhansError) as ei:
            fn(*args, **kw)
        return ei.value.code

    assert code(sn.stream_open, None, [synth.noise_clip(70, seconds=1.0)], [1000]) == -4     # < 200 context frames
    assert code(sn.stream_open, None, [neg], [-1]) == -2                                      # negative peak
    [sid] = sn.stream_open(None, [neg], [_peak(sn, mix)])
    assert code(sn.stream_step, [sid + 1000], [mix[:10]]) == -2                               # unknown id
    assert code(sn.stream_step, [sid, sid], [mix[:10], mix[10:20]]) == -2                     # the same id twice
    got = _stream_continue(sn, sid, mix)
    assert np.array_equal(got[0], want["i16"][0]) and np.array_equal(got[1], want["f32"][0])
    assert code(sn.stream_step, [sid], [mix[:10]]) == -2                                      # a chunk after the final step
    sn.stream_close([sid])
    assert code(sn.stream_step, [sid], [mix[:10]]) == -2                                      # closed id
    assert code(sn.stream_close, [sid]) == -2
    bare = Engine(0, 0, win_capacity=8, row_capacity=1)
    try:
        assert code(bare.stream_open, None, [neg], [1000]) == -3                              # weights not loaded
    finally:
        bare.close()
    # a weight reload closes the open streams, and ids go on counting: an id from before it never names a new stream
    small = _engine(W.SELECTIVE_NOISE, weights_sn, 8)
    try:
        [old] = small.stream_open(None, [neg], [1000])
        small.load_weights(weights_sn)
        assert code(small.stream_step, [old], [mix[:10]]) == -2
        [new] = small.stream_open(None, [neg], [1000])
        assert new > old
    finally:
        small.close()
    # the context still works: a fresh stream and the batch path
    _assert_equal(_stream(sn, mix, None, neg, [5000, 0, 1234, len(mix) - 6234]), want)
    assert np.array_equal(sn.enhance([mix], None, [neg])["i16"][0], want["i16"][0])


def _stream_continue(eng, sid, mix):
    r1 = eng.stream_step([sid], [mix[:7000]])
    r2 = eng.stream_step([sid], [mix[7000:]], final=[1])
    return np.concatenate([r1["i16"][0], r2["i16"][0]]), np.concatenate([r1["f32"][0], r2["f32"][0]])
