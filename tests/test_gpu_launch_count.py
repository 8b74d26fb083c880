"""nhans_profile_get kind 5 counts every kernel a stage-level entry point launches, profiling on or off."""
import numpy as np
import pytest

from nhans_b200 import synth

pytestmark = pytest.mark.gpu


def _launches(eng, call):
    eng.profile_reset()
    call()
    return eng.profile_get(5)["launches"]


def test_stage_entry_points_count_every_launch(engine_sn):
    eng = engine_sn
    clips = [synth.mixture(0.3, 0)[:400 + 160 * 5], synth.mixture(0.3, 1)[:400 + 160 * 2]]     # 6 + 3 frames
    lm, ph, fo, peak = eng.stft(clips)
    assert _launches(eng, lambda: eng.stft(clips)) == 2                                        # peaks + STFT
    assert _launches(eng, lambda: eng.stft_f32([c / np.float32(32768) for c in clips])) == 1
    assert _launches(eng, lambda: eng.normalise(clips)) == 2                                   # peaks + normalise
    assert _launches(eng, lambda: eng.eval_loss(lm, lm)) == 1
    assert _launches(eng, lambda: eng.istft(lm, ph, fo, peak=peak, want_i16=True)) == 1
    emb = np.random.default_rng(0).normal(0, 1, (2, 512)).astype(np.float32)
    # one pass of 9 windows: conditioning table, unit table, per-frame first convolution (the first GEMM layer builds its
    # operand from that table), one launch per GEMM layer, and the reduction of the split-K head
    n_gemm = len(eng.plan(0)["gemm"])
    assert _launches(eng, lambda: eng.masknet(lm, fo, emb, emb)) == 3 + n_gemm + 1
