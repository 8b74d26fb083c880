"""Host logic of the CLIs' live mode (--stream) that needs no GPU: raw PCM read in short and odd-sized pieces is handed to the
engine unchanged, the stream is flushed with an empty final step at EOF, the output bytes are exactly the engine's step
outputs, and the arguments a live stream cannot honour are rejected.  A fake engine stands in through get_engine."""
import io
import os
import sys

import numpy as np
import pytest

from nhans_b200 import synth
from nhans_b200.selective_noise import apply as sn_apply
from nhans_b200.source_separation import apply as ss_apply
from nhans_b200.wavio import write_wav


class _FakeStreams:
    """Records what the CLI feeds the streaming entry points; each step returns samples derived from its chunk."""

    def __init__(self):
        self.opened, self.steps, self.closed, self.returned = [], [], [], []

    def stream_open(self, ctx_a, ctx_b, peaks):
        self.opened.append((ctx_a, ctx_b, list(peaks)))
        return [7]

    def _out(self, chunk, final):
        # a final step emits the held-back tail; values beyond +-1 exercise the int16 saturation
        y = np.linspace(-1.5, 1.5, 11).astype(np.float32) if final else chunk.astype(np.float32) * np.float32(1e-4)
        self.returned.append(y)
        return y

    def stream_step_post(self, ids, chunks, compensate, final=None):
        assert ids == [7] and len(chunks) == 1 and chunks[0].dtype == np.int16
        self.steps.append(("post", chunks[0].copy(), compensate, final[0]))
        return {"compensated": [self._out(chunks[0], final[0])], "snr_est": np.ones(1, np.float32)}

    def stream_step(self, ids, chunks, final=None, want_f32=True, want_i16=True):
        assert ids == [7] and len(chunks) == 1 and chunks[0].dtype == np.int16
        self.steps.append(("plain", chunks[0].copy(), None, final[0]))
        y = self._out(chunks[0], final[0])
        return {"f32": [y] if want_f32 else None, "i16": [sn_apply._to_i16(y, 1000)] if want_i16 else None}

    def stream_close(self, ids):
        self.closed.append(list(ids))


@pytest.fixture
def wavs(tmp_path):
    write_wav(str(tmp_path / "neg.wav"), synth.noise_clip(3))
    write_wav(str(tmp_path / "pos.wav"), synth.noise_clip(3, "pos"))
    write_wav(str(tmp_path / "stereo.wav"), np.stack([synth.noise_clip(3), synth.noise_clip(4)], axis=1))
    return tmp_path


def _odd_reads(monkeypatch, sizes, limit):
    """os.read returns pieces of the given sizes (then whatever is asked), as a slow pipe would; every request is at
    most `limit` bytes."""
    real, it = os.read, iter(sizes)
    asked = []

    def read(fd, n):
        asked.append(n)
        assert n <= limit
        return real(fd, min(n, next(it, n)))
    monkeypatch.setattr(os, "read", read)
    return asked


def _pcm(n, seed=0):
    return np.random.default_rng(seed).integers(-32768, 32768, n).astype(np.int16)


def test_denoiser_stream_odd_reads_stdin_to_stdout(wavs, monkeypatch):
    x = _pcm(3001)
    raw = x.astype("<i2").tobytes()
    (wavs / "in.raw").write_bytes(raw)
    fake = _FakeStreams()
    monkeypatch.setattr(sn_apply, "get_engine", lambda v: fake)
    asked = _odd_reads(monkeypatch, [1, 3, 2, 5, 7, 1, 1, 64, 33], limit=2 * 16 * 3)
    out = io.BytesIO()
    with open(str(wavs / "in.raw"), "rb") as stdin:
        monkeypatch.setattr(sys, "stdin", stdin)
        monkeypatch.setattr(sys, "stdout", type("Out", (), {"buffer": out})())
        assert sn_apply.main(["--stream", "--input", "-", "--output", "-", "--neg", str(wavs / "neg.wav"),
                              "--compensate", "0.3", "--peak", "1234", "--chunk-ms", "3"]) == 0
    assert len(asked) > 20
    # Silent --pos (the default), the --neg clip, the given peak; one stream, closed at the end
    (ctx_a, ctx_b, peaks), = fake.opened
    assert ctx_a is None and np.array_equal(ctx_b[0], synth.noise_clip(3)) and peaks == [1234]
    assert fake.closed == [[7]]
    kinds = [s[0] for s in fake.steps]
    assert set(kinds) == {"post"} and all(s[2] == pytest.approx(0.3) for s in fake.steps)
    # every sample arrives once, in order, split wherever the reads fell; no empty step before EOF
    assert np.array_equal(np.concatenate([s[1] for s in fake.steps]), x)
    assert all(len(s[1]) > 0 and not s[3] for s in fake.steps[:-1])
    assert len(fake.steps[-1][1]) == 0 and fake.steps[-1][3] == 1
    # reads of 1, 3, 2, 5, 7, 1, 1, 64, 33 bytes: an odd byte waits for the next read, a lone byte makes no step
    assert [len(s[1]) for s in fake.steps[:7]] == [2, 1, 2, 4, 1, 32, 16]
    want = b"".join(sn_apply._to_i16(y, 1234).astype("<i2").tobytes() for y in fake.returned)
    assert out.getvalue() == want


def test_denoiser_stream_files_float32_and_trailing_byte(wavs, monkeypatch, capsys):
    x = _pcm(1000, 1)
    (wavs / "in.raw").write_bytes(x.astype("<i2").tobytes() + b"\x01")       # an incomplete last sample
    fake = _FakeStreams()
    monkeypatch.setattr(sn_apply, "get_engine", lambda v: fake)
    assert sn_apply.main(["--stream", "--input", str(wavs / "in.raw"), "--output", str(wavs / "out.raw"),
                          "--neg", str(wavs / "neg.wav"), "--pos", str(wavs / "pos.wav"), "--float32"]) == 0
    assert np.array_equal(fake.opened[0][0][0], synth.noise_clip(3, "pos")) and fake.opened[0][2] == [32767]
    assert np.array_equal(np.concatenate([s[1] for s in fake.steps]), x)
    assert fake.steps[-1][3] == 1 and len(fake.steps[-1][1]) == 0
    assert all(s[2] == 0.0 for s in fake.steps)
    assert (wavs / "out.raw").read_bytes() == b"".join(y.astype("<f4").tobytes() for y in fake.returned)
    assert "odd trailing byte" in capsys.readouterr().err


def test_denoiser_int16_rule_saturates(wavs, monkeypatch):
    (wavs / "in.raw").write_bytes(b"")
    fake = _FakeStreams()
    monkeypatch.setattr(sn_apply, "get_engine", lambda v: fake)
    sn_apply.main(["--stream", "--input", str(wavs / "in.raw"), "--output", str(wavs / "out.raw"), "--neg", str(wavs / "neg.wav")])
    assert [s[3] for s in fake.steps] == [1]                                  # only the empty final step
    got = np.frombuffer((wavs / "out.raw").read_bytes(), "<i2")
    assert got[0] == -32768 and got[-1] == 32767
    assert np.array_equal(got, np.clip(np.rint(fake.returned[0] * np.float32(32767.000001)), -32768, 32767))


def _rejected(main, argv, capsys):
    with pytest.raises(SystemExit) as ei:
        main(argv)
    assert ei.value.code == 2
    return capsys.readouterr().err


def test_ac_with_stream_is_rejected(wavs, monkeypatch, capsys):
    fake = _FakeStreams()
    monkeypatch.setattr(sn_apply, "get_engine", lambda v: fake)
    err = _rejected(sn_apply.main, ["--stream", "--ac", "--input", "-", "--output", "-", "--neg", str(wavs / "neg.wav")], capsys)
    assert "--ac" in err and "snr_est" in err
    assert not fake.opened


@pytest.mark.parametrize("flag", ["--neg", "--pos"])
def test_stereo_context_is_rejected(wavs, monkeypatch, capsys, flag):
    fake = _FakeStreams()
    monkeypatch.setattr(sn_apply, "get_engine", lambda v: fake)
    monkeypatch.setattr(ss_apply, "get_engine", lambda v: fake)
    ctx = {"--neg": str(wavs / "neg.wav"), "--pos": str(wavs / "pos.wav")}
    ctx[flag] = str(wavs / "stereo.wav")
    argv = ["--stream", "--input", "-", "--output", "-", "--neg", ctx["--neg"], "--pos", ctx["--pos"]]
    for main in (sn_apply.main, ss_apply.main):
        err = _rejected(main, argv, capsys)
        assert flag in err and "int16 mono" in err
    assert not fake.opened


def test_bad_peak_and_chunk_are_rejected(wavs, capsys):
    base = ["--stream", "--input", "-", "--output", "-", "--neg", str(wavs / "neg.wav")]
    assert "--peak" in _rejected(sn_apply.main, base + ["--peak", "-1"], capsys)
    assert "--chunk-ms" in _rejected(sn_apply.main, base + ["--chunk-ms", "0"], capsys)


def test_separator_stream_uses_the_plain_step(wavs, monkeypatch):
    x = _pcm(2500, 2)
    (wavs / "in.raw").write_bytes(x.astype("<i2").tobytes())
    fake = _FakeStreams()
    monkeypatch.setattr(ss_apply, "get_engine", lambda v: fake)
    _odd_reads(monkeypatch, [5, 1, 1, 1, 9], limit=2 * 16 * 100)
    assert ss_apply.main(["--stream", "--input", str(wavs / "in.raw"), "--output", str(wavs / "out.raw"),
                          "--neg", str(wavs / "neg.wav"), "--pos", str(wavs / "pos.wav"), "--peak", "1000"]) == 0
    (ctx_a, ctx_b, peaks), = fake.opened
    assert np.array_equal(ctx_a[0], synth.noise_clip(3)) and np.array_equal(ctx_b[0], synth.noise_clip(3, "pos"))   # a = --neg
    assert peaks == [1000] and fake.closed == [[7]]
    assert {s[0] for s in fake.steps} == {"plain"}
    assert np.array_equal(np.concatenate([s[1] for s in fake.steps]), x)
    assert fake.steps[-1][3] == 1 and len(fake.steps[-1][1]) == 0
    want = b"".join(sn_apply._to_i16(y, 1000).astype("<i2").tobytes() for y in fake.returned)
    assert (wavs / "out.raw").read_bytes() == want
