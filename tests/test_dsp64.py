"""The float64 references of tests/dsp64.py agree with the oracle's STFT, inverse STFT, int16 conversion and post-mix,
so that the GPU edge tests (test_gpu_dsp_edges.py) rest on references that are checked without a GPU."""
import numpy as np

import dsp64 as R
from nhans_b200 import synth
from oracle import nhans_oracle as O


def test_references_match_oracle():
    rng = np.random.default_rng(0)
    for n in (0, 399, 400, 401, 559, 560, 4000 + 79):
        pcm = synth.mixture(0.3, n % 7)[:n].copy()
        if n:
            pcm[n // 2] = -32768
        x = O.normalise(pcm)
        X = R.stft64(x)
        assert X.shape == (O.frame_index(n).shape[0], 201)
        assert np.array_equal(X, O.stft(x))                      # same frames, window and transform
        if n:
            xr = R.normalise_i16(pcm)
            assert np.abs(xr.astype(np.float64) - x).max() <= np.abs(x).max() * 2.0 ** -23   # reciprocal vs true quotient
        lm = rng.normal(-2, 2, X.shape).astype(np.float32)
        ph = rng.uniform(-np.pi, np.pi, X.shape).astype(np.float32)
        y = R.istft64(np.exp(lm.astype(np.float64)), np.exp(1j * ph.astype(np.float64)))
        yo = O.istft(lm, ph)
        assert len(y) == len(yo) == (O.trim_len(n) if n >= 400 else 0)
        if len(y):
            assert np.abs(y - yo).max() <= 1e-6 * np.abs(y).max()
    # the STFT -> iSTFT identity of the float64 pair (away from the edges, which fewer than three frames cover)
    x = O.normalise(synth.mixture(0.5, 3))[:O.trim_len(8000)]
    X = R.stft64(x)
    assert np.abs(R.istft64(np.abs(X), np.exp(1j * np.angle(X))) - x)[400:-400].max() < 1e-12


def test_i16_rule_and_postmix_match_oracle():
    rng = np.random.default_rng(1)
    y = np.concatenate([rng.uniform(-1.6, 1.6, 5000), [1.0, -1.0, 0.5 / 32767, 1.5 / 32767, -2.5 / 32767]]).astype(np.float32)
    for peak in (0, 1, 1000, 32767, -32768):
        got = R.i16_rule(y, peak)
        assert np.array_equal(got, O.to_int16(y, float(peak)))
        if peak == 32767:
            assert got.max() == 32767 and got.min() == -32768          # both ends saturate
    den = rng.normal(0, 0.3, 3000).astype(np.float32)
    mixed = (den + rng.normal(0, 0.1, 3000)).astype(np.float32)
    for ac, comp in ((False, 0.3), (True, 0.0)):
        removed, snr, compensated, _ = R.postmix64(den, mixed, comp, ac)
        r_o, snr_o, c_o = O.post_mix(den, mixed, comp, ac)
        assert np.array_equal(removed, r_o)
        assert abs(snr - snr_o) <= 1e-6 * snr_o                    # the oracle averages in float32
        assert np.abs(compensated - c_o).max() <= 1e-6 * np.abs(c_o).max()
    removed, snr, compensated, factor = R.postmix64(np.zeros(0, np.float32), np.zeros(0, np.float32), 0.0, True)
    assert snr == np.inf and factor == 0 and removed.size == compensated.size == 0
