"""Emission rule of streaming enhancement (nhans_stream_emit_len, host only): what a stream has emitted after N samples
follows from frames_of(N) alone, whatever the chunking, and after the final step it is the batch path's output length."""
import ctypes

import numpy as np

from nhans_b200 import _lib


def _frames(n):
    return 1 + (n - 400) // 160 if n >= 400 else 0


def _out_len(F):
    return (F - 1) * 160 + 400 if F > 0 else 0


def _emit(before, after, final):
    e = ctypes.c_int64()
    assert _lib.load().nhans_stream_emit_len(before, after, int(final), ctypes.byref(e)) == 0
    return e.value


def test_emitted_lengths_follow_the_rule_for_random_chunkings():
    rng = np.random.default_rng(0)
    sizes = [0, 1, 159, 160, 161, 399, 400, 1600, 2960, 7919]
    for trial in range(300):
        total = int(rng.integers(0, 160001)) if trial % 3 else int(rng.integers(0, 400))
        n = emitted = 0
        while True:
            step = int(rng.choice(sizes)) if trial % 2 else int(rng.integers(0, 4000))
            step = min(step, total - n)
            final = n + step == total and rng.random() < 0.7
            e = _emit(n, n + step, final)
            assert e >= 0 and e % (80 if final else 160) == 0
            n += step
            emitted += e
            if final:
                assert emitted == _out_len(_frames(n)) == _out_len(_frames(total))
                break
            # the non-final total: every hop whose three frames' windows have their 17 right-hand frames
            assert emitted == 160 * max(0, _frames(n) - 17)
            if _frames(n) < 18:
                assert emitted == 0
            if n == total and step == 0:           # everything delivered: an empty final step flushes the rest
                assert _emit(n, n, True) == _out_len(_frames(n)) - emitted
                break


def test_emit_len_edges_and_argument_errors():
    assert _emit(0, 399, True) == 0                 # no frame: the batch path returns nothing either
    assert _emit(0, 400, True) == 400
    assert _emit(0, 400 + 16 * 160, False) == 0     # 17 frames: no window has its look-ahead yet
    assert _emit(0, 400 + 17 * 160, False) == 160   # 18 frames: the first hop
    assert _emit(0, 400 + 17 * 160 + 159, False) == 160
    e = ctypes.c_int64()
    lib = _lib.load()
    assert lib.nhans_stream_emit_len(10, 5, 0, ctypes.byref(e)) != 0
    assert lib.nhans_stream_emit_len(-1, 5, 0, ctypes.byref(e)) != 0
    assert lib.nhans_stream_emit_len(0, 5, 0, None) != 0
