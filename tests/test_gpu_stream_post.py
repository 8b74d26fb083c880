"""Post-mix outputs of live streams (nhans_stream_step_post): for every chunking and compensate factor, a stream's
concatenated denoised, mixed_processed, removed and compensated samples equal the batch path's (enhance + nhans_postmix with
ac = 0) bit for bit; its running snr_est follows the float64 ratio of the energy it has emitted; the batch path is
undisturbed; and the CLIs' --stream mode reproduces the batch int16 output byte for byte through a pipe."""
import os
import subprocess
import sys

import numpy as np
import pytest

import dsp64 as R
from nhans_b200 import synth, weights as W
from nhans_b200.engine import Engine, NhansError, pack
from nhans_b200.wavio import write_wav

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RANDOM_SIZES = [0, 1, 159, 160, 161, 399, 400, 2960, 7919]
# < 400 samples, 20 frames, 40 frames (+ a partial hop), 4 s
LENGTHS = [300, 400 + 19 * 160, 400 + 39 * 160 + 77, 64000]
COMPENSATE = [0.0, 0.3, -0.7]
POST_KEYS = ("mixed_processed", "removed", "compensated")
SNR_BOUND = 2e-7                # relative; the float64 sums of the batch path are grouped differently
_snr_max = [0.0]                # largest relative snr_est error seen, printed when the module ends


@pytest.fixture(scope="module", autouse=True)
def _report_snr_maximum():
    yield
    print("\nstream snr_est: largest relative error %.3g (bound %.1g)" % (_snr_max[0], SNR_BOUND))


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


def _ratio64(den, removed):
    e_den = float(np.sum(np.asarray(den, np.float64) ** 2))
    e_rem = float(np.sum(np.asarray(removed, np.float64) ** 2))
    return e_den / e_rem if e_rem > 0 else np.inf


def _check_snr(got, want):
    if np.isinf(want):
        assert np.isinf(got) and got > 0, (got, want)
        return
    err = abs(float(got) - want) / abs(want)
    _snr_max[0] = max(_snr_max[0], err)
    assert err <= SNR_BOUND, (got, want)


def _batch(eng, mixes, ctx_a, ctx_b, comps):
    """enhance + one nhans_postmix(c, ac = 0) per compensate value c -> (enhance result, {c: postmix result})"""
    want = eng.enhance(mixes, ctx_a, ctx_b)
    return want, {c: eng.postmix(want["out_offs"], compensate=c) for c in comps}


def _stream_post(eng, mix, ctx_a, ctx_b, sizes, comp, empty_final=False):
    """Feed mix in chunks of `sizes` through post steps; checks the running snr_est after every step.
    -> dict of concatenated outputs and the last snr_est"""
    [sid] = eng.stream_open(None if ctx_a is None else [ctx_a], [ctx_b], [_peak(eng, mix)])
    steps = [(s, False) for s in sizes[:-1]] + [(sizes[-1] if sizes else 0, not empty_final)]
    if empty_final:
        steps.append((0, True))
    got = {k: [] for k in ("i16", "f32") + POST_KEYS}
    n, snr = 0, None
    for size, final in steps:
        r = eng.stream_step_post([sid], [mix[n:n + size]], comp, final=[int(final)])
        n += size
        for k in got:
            got[k].append(r[k][0])
        snr = float(r["snr_est"][0])
        _check_snr(snr, _ratio64(np.concatenate(got["f32"]), np.concatenate(got["removed"])))
    assert n == len(mix)
    eng.stream_close([sid])
    out = {k: np.concatenate(v) for k, v in got.items()}
    out["snr_est"] = snr
    return out


def _assert_bits(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8)), what


def _assert_matches(got, want, post, u, what):
    _assert_bits(got["i16"], want["i16"][u], what + " i16")
    _assert_bits(got["f32"], want["f32"][u], what + " f32")
    for k in POST_KEYS:
        _assert_bits(got[k], post[k][u], what + " " + k)


def _contexts(case, seed):
    if case == "sn_silent":
        return None, synth.noise_clip(seed)
    if case == "sn_pos_neg":
        return synth.noise_clip(seed, "pos"), synth.noise_clip(seed, "neg")
    return synth.speaker_clip(seed, "interference"), synth.speaker_clip(seed, "target")


@pytest.mark.parametrize("case", ["sn_silent", "sn_pos_neg", "ss"])
def test_stream_post_bit_identical_to_batch(case, sn, ss):
    rng = np.random.default_rng(11)
    eng = ss if case == "ss" else sn
    for li, length in enumerate(LENGTHS):
        mix = synth.mixture(4.2, 20 + li)[:length]
        ctx_a, ctx_b = _contexts(case, 20 + li)
        want, posts = _batch(eng, [mix], None if ctx_a is None else [ctx_a], [ctx_b], COMPENSATE)
        for kind, empty_final in (("one", False), ("1600", False), ("random", False), ("random", True)):
            for c in COMPENSATE:
                got = _stream_post(eng, mix, ctx_a, ctx_b, _chunking(kind, len(mix), rng), c, empty_final)
                what = "%s len %d %s%s c %g" % (case, length, kind, " + empty final" if empty_final else "", c)
                _assert_matches(got, want, posts[c], 0, what)
                if length < 400:
                    assert np.isinf(got["snr_est"]) and np.isinf(posts[c]["snr_est"][0])
                else:
                    _check_snr(got["snr_est"], float(posts[c]["snr_est"][0]))


def test_many_streams_ragged_lifetimes_own_compensate(weights_sn, sn):
    """40 streams, each with its own factor, open and finish at different steps on an engine whose passes hold 64 windows;
    each equals the batch post-mix of its clip for its factor, computed on an engine of another capacity."""
    rng = np.random.default_rng(12)
    eng = _engine(W.SELECTIVE_NOISE, weights_sn, 64)
    try:
        S = 40
        mixes = [synth.mixture(0.2 + 0.05 * (u % 9), 100 + u)[:int(rng.integers(300, 24000))] for u in range(S)]
        negs = [synth.noise_clip(100 + u % 4) for u in range(S)]
        comps = [float(np.float32(v)) for v in rng.uniform(-1.0, 1.0, S)]
        comps[0] = 0.0
        want, posts = _batch(sn, mixes, None, negs, sorted(set(comps)))
        opens = rng.integers(0, 12, S)
        ids, pos = {}, [0] * S
        outs = [{k: [] for k in ("i16", "f32") + POST_KEYS} for _ in range(S)]
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
            r = eng.stream_step_post([ids[u] for u in live], chunks, [comps[u] for u in live], final=finals)
            for k, u in enumerate(live):
                pos[u] += len(chunks[k])
                for key in outs[u]:
                    outs[u][key].append(r[key][k])
                _check_snr(r["snr_est"][k], _ratio64(np.concatenate(outs[u]["f32"]), np.concatenate(outs[u]["removed"])))
                if finals[k]:
                    eng.stream_close([ids[u]])
                    ids[u] = None
        assert len(ids) == S and all(v is None for v in ids.values())
        for u in range(S):
            got = {k: np.concatenate(v) for k, v in outs[u].items()}
            _assert_matches(got, want, posts[comps[u]], u, "stream %d c %g" % (u, comps[u]))
    finally:
        eng.close()


def test_snr_is_inf_before_the_first_sample(sn):
    mix, neg = synth.mixture(1.0, 80), synth.noise_clip(80)
    [sid] = sn.stream_open(None, [neg], [_peak(sn, mix)])
    r = sn.stream_step_post([sid], [mix[:2000]], 0.3)                        # 10 frames: nothing emitted yet
    assert len(r["f32"][0]) == 0 and np.isinf(r["snr_est"][0])
    r = sn.stream_step_post([sid], [mix[2000:]], 0.3, final=[1])
    assert np.isfinite(r["snr_est"][0])
    sn.stream_close([sid])


def test_nan_compensate_gives_the_denoised_signal(sn):
    mix, neg = synth.mixture(1.5, 81), synth.noise_clip(81)
    nan = float("nan")
    want, posts = _batch(sn, [mix], None, [neg], [nan])
    got = _stream_post(sn, mix, None, neg, _chunking("1600", len(mix), None), nan)
    assert np.array_equal(got["compensated"], got["f32"])
    _assert_matches(got, want, posts[nan], 0, "nan")


def test_plain_and_post_steps_mixed(sn):
    """Post-step outputs of a stream that also takes plain steps equal the matching slices of the batch outputs, and its
    snr_est covers only the samples of its post steps."""
    mix, neg = synth.mixture(3.0, 82), synth.noise_clip(82)
    want, posts = _batch(sn, [mix], None, [neg], [0.3])
    post = posts[0.3]
    [sid] = sn.stream_open(None, [neg], [_peak(sn, mix)])
    n, emitted, den, rem, post_steps = 0, 0, [], [], 0
    sizes = _chunking("1600", len(mix), None)
    for k, size in enumerate(sizes):
        final = [int(k == len(sizes) - 1)]
        if k % 3 == 1:
            r = sn.stream_step([sid], [mix[n:n + size]], final=final)
        else:
            r = sn.stream_step_post([sid], [mix[n:n + size]], 0.3, final=final)
            sl = slice(emitted, emitted + len(r["f32"][0]))
            for key in POST_KEYS:
                _assert_bits(r[key][0], post[key][0][sl], "step %d %s" % (k, key))
            den.append(r["f32"][0])
            rem.append(r["removed"][0])
            post_steps += len(r["f32"][0]) > 0
            _check_snr(r["snr_est"][0], _ratio64(np.concatenate(den), np.concatenate(rem)))
        _assert_bits(r["i16"][0], want["i16"][0][emitted:emitted + len(r["i16"][0])], "step %d i16" % k)
        _assert_bits(r["f32"][0], want["f32"][0][emitted:emitted + len(r["f32"][0])], "step %d f32" % k)
        n += size
        emitted += len(r["f32"][0])
    assert emitted == len(want["f32"][0]) and post_steps > 3
    sn.stream_close([sid])


def test_post_steps_leave_batch_results_alone(sn):
    A = ([synth.mixture(0.5, 60), synth.mixture(0.3, 61)], None, [synth.noise_clip(60), synth.noise_clip(61)])
    ref = sn.enhance(*A)
    post_ref = sn.postmix(ref["out_offs"], compensate=0.3)
    mix, neg = synth.mixture(1.0, 62), synth.noise_clip(62)
    [sid] = sn.stream_open(None, [neg], [32767])
    # a post step while a submitted batch is in flight
    t = sn.submit(*A)
    sn.stream_step_post([sid], [mix[:8000]], 0.6)
    got = sn.collect(t)
    for u in range(2):
        assert np.array_equal(got["i16"][u], ref["i16"][u]) and np.array_equal(got["f32"][u], ref["f32"][u])
    # a post step between run and postmix / download
    m, mo = pack(A[0])
    b, bo = pack(A[2])
    sn.upload(m, mo, None, None, b, bo)
    sn.run()
    sn.stream_step_post([sid], [mix[8000:]], -0.2, final=[1])
    n = int(ref["out_offs"][-1])
    o16, o32 = np.zeros(n, np.int16), np.zeros(n, np.float32)
    sn.download(o16, o32)
    sn.sync()
    assert np.array_equal(o16, np.concatenate(ref["i16"])) and np.array_equal(o32, np.concatenate(ref["f32"]))
    post = sn.postmix(ref["out_offs"], compensate=0.3)
    for k in POST_KEYS:
        for u in range(2):
            _assert_bits(post[k][u], post_ref[k][u], k)
    _assert_bits(post["snr_est"], post_ref["snr_est"], "snr_est")
    sn.stream_close([sid])


def test_post_step_argument_errors(sn):
    mix, neg = synth.mixture(0.6, 70), synth.noise_clip(70)

    def code(*args, **kw):
        with pytest.raises(NhansError) as ei:
            sn.stream_step_post(*args, **kw)
        return ei.value.code

    [sid] = sn.stream_open(None, [neg], [_peak(sn, mix)])
    assert code([sid + 1000], [mix[:10]], 0.0) == -2                                       # unknown id
    assert code([sid, sid], [mix[:10], mix[10:20]], [0.0, 0.0]) == -2                      # the same id twice
    sn.stream_step_post([sid], [mix], 0.0, final=[1])
    assert code([sid], [mix[:10]], 0.0) == -2                                              # a chunk after the final step
    sn.stream_close([sid])
    assert code([sid], [mix[:10]], 0.0) == -2                                              # closed id
    bare = Engine(0, 0, win_capacity=8, row_capacity=1)
    try:
        with pytest.raises(NhansError) as ei:
            bare.stream_step_post([0], [mix[:10]], 0.0)
        assert ei.value.code == -3                                                         # weights not loaded
    finally:
        bare.close()


def _cli(module, args, stdin, tmp_path):
    env = dict(os.environ, NHANS_ALLOW_RANDOM_INIT="1", NHANS_SEED="0", NHANS_MODEL_DIR=str(tmp_path / "no_model"),
               PYTHONPATH=ROOT)
    os.makedirs(str(tmp_path / "no_model"), exist_ok=True)
    p = subprocess.run([sys.executable, "-m", module, "--stream", "--input", "-", "--output", "-", "--chunk-ms", "37"] + args,
                       input=stdin, capture_output=True, cwd=ROOT, env=env, timeout=600)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    return p.stdout


def test_cli_denoiser_stream_round_trip(sn, tmp_path):
    mix, neg = synth.mixture(4.0, 90), synth.noise_clip(90)
    write_wav(str(tmp_path / "neg.wav"), neg)
    P = _peak(sn, mix)
    want, posts = _batch(sn, [mix], None, [neg], [0.3])
    out = _cli("nhans_b200.selective_noise.apply", ["--neg", str(tmp_path / "neg.wav"), "--peak", str(P), "--compensate", "0.3"],
               mix.astype("<i2").tobytes(), tmp_path)
    assert out == R.i16_rule(posts[0.3]["compensated"][0], P).astype("<i2").tobytes()


def test_cli_separator_stream_round_trip(ss, tmp_path):
    mix = synth.mixture(4.0, 91)
    interference, target = synth.speaker_clip(91, "interference"), synth.speaker_clip(91, "target")
    write_wav(str(tmp_path / "neg.wav"), interference)
    write_wav(str(tmp_path / "pos.wav"), target)
    P = _peak(ss, mix)
    want = ss.enhance([mix], [interference], [target])
    out = _cli("nhans_b200.source_separation.apply", ["--neg", str(tmp_path / "neg.wav"), "--pos", str(tmp_path / "pos.wav"),
                                                      "--peak", str(P)], mix.astype("<i2").tobytes(), tmp_path)
    assert out == want["i16"][0].astype("<i2").tobytes()
