"""Host-side driver of one GPU context (one per GPU, one thread each): thin numpy <-> C-ABI glue.

Everything numerical happens inside libnhans_b200.so; this module only marshals arrays, concatenates
ragged utterance lists into (data, offsets) pairs and owns pinned staging buffers."""
from __future__ import annotations

import ctypes
import json

import numpy as np

from . import _lib, weights as W

N_BINS = 201
CTX_FRAMES = 200
KIND_GEMM, KIND_STFT, KIND_ISTFT, KIND_DIRECT, KIND_OTHER = range(5)
STREAM_EMIT_SLACK = 17 * 160 + 400


class NhansError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libnhans_b200 error %d: %s" % (code, msg))
        self.code = code


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def pack(clips, dtype=np.int16, alloc=np.empty):
    """List of 1-D arrays -> (concatenated `dtype` samples, int64 offsets [U+1]).  `alloc(n, dtype)` provides the
    contiguous array the samples are copied into."""
    offs = np.zeros(len(clips) + 1, np.int64)
    for i, c in enumerate(clips):
        offs[i + 1] = offs[i] + len(c)
    data = alloc(int(offs[-1]), dtype)
    for i, c in enumerate(clips):
        data[offs[i]:offs[i + 1]] = c
    return data, offs


def unpack(data, offs):
    return [data[offs[i]:offs[i + 1]] for i in range(len(offs) - 1)]


class PinnedArray:
    """numpy view over cudaHostAlloc memory (asynchronous H2D / D2H copies need it)."""

    def __init__(self, shape, dtype):
        self.lib = _lib.load()
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = ctypes.c_void_p()
        rc = self.lib.nhans_host_alloc(max(self.nbytes, 1), ctypes.byref(p))
        if rc:
            raise NhansError(rc, "cudaHostAlloc failed")
        self.ptr = p
        buf = (ctypes.c_char * max(self.nbytes, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if self.ptr:
            self.array = None
            self.lib.nhans_host_free(self.ptr)
            self.ptr = None


class Engine:
    def __init__(self, device=0, variant=W.SELECTIVE_NOISE, win_capacity=0, row_capacity=0):
        self.lib = _lib.load()
        self.variant = variant
        self.device = device
        h = ctypes.c_void_p()
        rc = self.lib.nhans_create(device, variant, win_capacity, row_capacity, ctypes.byref(h))
        if rc:
            raise NhansError(rc, self.lib.nhans_last_error(None).decode())
        self.h = h
        self.weight_source = None

    # ------------------------------------------------------------------------------------------
    def _ck(self, rc):
        if rc:
            raise NhansError(rc, self.lib.nhans_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.nhans_destroy(self.h)
            self.h = None
            for pool in self.__dict__.get("_stage_bufs", []):
                for buf in pool.values():
                    buf.free()
            self.__dict__.pop("_stage_bufs", None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def load_weights(self, weights, source="array"):
        names = sorted(weights)
        arrs = [np.ascontiguousarray(weights[n], dtype=np.float32) for n in names]
        c_names = (ctypes.c_char_p * len(names))(*[n.encode() for n in names])
        c_sizes = (ctypes.c_int64 * len(names))(*[a.size for a in arrs])
        c_data = (ctypes.c_void_p * len(names))(*[a.ctypes.data for a in arrs])
        self._ck(self.lib.nhans_load_weights(self.h, c_names, c_sizes, c_data, len(names)))
        self.weight_source = source

    def load_default_weights(self, model_dir=None, seed=0, allow_random=None):
        w, src = W.load_or_init(self.variant, model_dir, seed, allow_random)
        self.load_weights(w, src)
        return src

    # ---- stage-level --------------------------------------------------------------------------
    def normalise(self, clips, trim=True):
        data, offs = pack(clips)
        out = np.zeros(int(offs[-1]), np.float32)
        out_offs = np.zeros(len(clips) + 1, np.int64)
        self._ck(self.lib.nhans_normalise(self.h, _ptr(data), _ptr(offs), len(clips), int(trim), _ptr(out), _ptr(out_offs)))
        return [out[out_offs[i]:out_offs[i + 1]] for i in range(len(clips))]

    def stft(self, clips):
        """-> (logmag [F,201], phase [F,201], frame_offs [U+1], peak [U])"""
        data, offs = pack(clips)
        U = len(clips)
        fo = np.zeros(U + 1, np.int64)
        self._ck(self.lib.nhans_stft(self.h, _ptr(data), _ptr(offs), U, None, None, _ptr(fo), None))
        F = int(fo[-1])
        lm = np.zeros((F, N_BINS), np.float32)
        ph = np.zeros((F, N_BINS), np.float32)
        peak = np.zeros(U, np.int32)
        self._ck(self.lib.nhans_stft(self.h, _ptr(data), _ptr(offs), U, _ptr(lm), _ptr(ph), _ptr(fo), _ptr(peak)))
        return lm, ph, fo, peak

    def stft_f32(self, signals):
        """float32 sample arrays (already normalised / mixed) -> (logmag [F,201], phase [F,201], frame_offs [U+1])"""
        U = len(signals)
        data, offs = pack(signals, np.float32)
        fo = np.zeros(U + 1, np.int64)
        self._ck(self.lib.nhans_stft_f32(self.h, _ptr(data), _ptr(offs), U, None, None, _ptr(fo)))
        F = int(fo[-1])
        lm = np.zeros((F, N_BINS), np.float32)
        ph = np.zeros((F, N_BINS), np.float32)
        self._ck(self.lib.nhans_stft_f32(self.h, _ptr(data), _ptr(offs), U, _ptr(lm), _ptr(ph), _ptr(fo)))
        return lm, ph, fo

    def enhance_f32(self, mixes, ctx_a, ctx_b, start=0, want_mixproc=True):
        """Fused float path (nhans_enhance_f32): lists of float sample arrays that are already normalised / mixed on the
        host; contexts = first 200 frames of ctx_a[u] / ctx_b[u] (ctx_a may be None: Silent.wav); the mask network runs
        over mixture frames [start:].  One device pass, no host round trips between the stages.
        -> (list of denoised sample arrays, list of mixture-centre sample arrays or None)"""
        m, mo = pack(mixes, np.float32)
        b, bo = pack(ctx_b, np.float32)
        a, ao = pack(ctx_a, np.float32) if ctx_a is not None else (None, None)
        U = len(mixes)
        oo = np.zeros(U + 1, np.int64)
        self._ck(self.lib.nhans_enhance_f32(self.h, _ptr(m), _ptr(mo), U, _ptr(a), _ptr(ao), _ptr(b), _ptr(bo), int(start), None, None, _ptr(oo)))
        y = np.zeros(int(oo[-1]), np.float32)
        ym = np.zeros(int(oo[-1]), np.float32) if want_mixproc else None
        self._ck(self.lib.nhans_enhance_f32(self.h, _ptr(m), _ptr(mo), U, _ptr(a), _ptr(ao), _ptr(b), _ptr(bo), int(start), _ptr(y), _ptr(ym), _ptr(oo)))
        return unpack(y, oo), (unpack(ym, oo) if want_mixproc else None)

    def enhance_demo(self, mix, sig_a, sig_b, start=CTX_FRAMES):
        """apply_demo (SN/apply.py:247-337, SS/apply.py:198-285): float mixture + two float context signals.
        Contexts are the first 200 frames of sig_a / sig_b, windows are taken over mix frames [start:] only (the
        slice is zero padded like a whole utterance).  -> (denoised samples, mixture-centre samples)."""
        y, ymix = self.enhance_f32([mix], [sig_a], [sig_b], start=start)
        return y[0], ymix[0]

    def enhance_float(self, mix, ctx_a, ctx_b):
        """apply_snc / apply_separator for clips that are not int16 PCM (stereo files averaged in float64,
        SN/apply.py:46-53): host normalisation exactly like handle_signals (SN/apply.py:142-163), then the fused float
        entry point.  ctx_a may be None (Silent.wav).  -> dict(f32=denoised samples, mixed_processed=..., peak=max|mix|)."""
        from .wavio import normalise_host
        m = normalise_host(mix)
        if len(m) >= 400:
            m = m[:len(m) - (len(m) - 400) % 160]
        x = np.asarray(mix)
        peak = float(max(abs(x))) if len(x) else 0.0
        if len(m) < 400:
            z = np.zeros(0, np.float32)
            return dict(f32=z, mixed_processed=z, peak=peak)
        y, ymix = self.enhance_f32([m], None if ctx_a is None else [normalise_host(ctx_a)], [normalise_host(ctx_b)], start=0)
        return dict(f32=y[0], mixed_processed=ymix[0], peak=peak)

    def eval_loss(self, denoised, target):
        """example_loss of the model graph (SN/main.py:243-246): [n,201] x [n,201] -> [n]."""
        d = np.ascontiguousarray(denoised, np.float32).reshape(-1, N_BINS)
        t = np.ascontiguousarray(target, np.float32).reshape(-1, N_BINS)
        assert d.shape == t.shape
        out = np.zeros(d.shape[0], np.float32)
        self._ck(self.lib.nhans_eval_loss(self.h, _ptr(d), _ptr(t), d.shape[0], _ptr(out)))
        return out

    def eval_outputs(self, mixed, target, sig_a, sig_b, extra=(), start=CTX_FRAMES):
        """Eval-mode example stream + model outputs for one seed tuple (SN/reader.py:398-420 + SN/main.py:231-252):
        STFT of the float signals, contexts = first 200 frames of sig_a / sig_b, frames [start:] of the mixture
        through the mask network, per-frame loss against the target's log-magnitude.  ``extra`` signals are only
        transformed (their log-magnitude / phase rows [start:] are returned, e.g. the SN pos / neg references)."""
        sigs = [mixed, target, sig_a, sig_b] + list(extra)
        lm, ph, fo = self.stft_f32(sigs)
        T = int(fo[1])
        for u in (2, 3):
            if fo[u + 1] - fo[u] < CTX_FRAMES:
                raise NhansError(-4, "context signal yields %d < 200 STFT frames" % (fo[u + 1] - fo[u]))
        if T <= start or fo[2] - fo[1] != T:
            raise NhansError(-2, "mixture / target frame counts %d / %d (need > %d and equal)" % (T, fo[2] - fo[1], start))
        emb = self.embed(np.stack([lm[fo[2]:fo[2] + CTX_FRAMES], lm[fo[3]:fo[3] + CTX_FRAMES]]))
        sl = np.ascontiguousarray(lm[start:T])
        den = self.masknet(sl, np.array([0, T - start], np.int64), emb[0:1], emb[1:2])
        tgt = np.ascontiguousarray(lm[fo[1] + start:fo[2]])
        out = dict(loss=self.eval_loss(den, tgt), mixed=sl, denoised=den, mixedph=np.ascontiguousarray(ph[start:T]),
                   target=tgt, targetph=np.ascontiguousarray(ph[fo[1] + start:fo[2]]),
                   location=np.arange(T - start, dtype=np.int32))
        out["extra"] = [(np.ascontiguousarray(lm[fo[4 + i] + start:fo[5 + i]]), np.ascontiguousarray(ph[fo[4 + i] + start:fo[5 + i]]))
                        for i in range(len(extra))]
        return out

    def embed(self, ctx_logmag):
        x = np.ascontiguousarray(ctx_logmag, np.float32).reshape(-1, CTX_FRAMES, N_BINS)
        emb = np.zeros((x.shape[0], 512), np.float32)
        self._ck(self.lib.nhans_embed(self.h, _ptr(x), x.shape[0], _ptr(emb)))
        return emb

    def masknet(self, logmag, frame_offs, emb_a, emb_b):
        lm = np.ascontiguousarray(logmag, np.float32)
        fo = np.ascontiguousarray(frame_offs, np.int64)
        ea = np.ascontiguousarray(emb_a, np.float32)
        eb = np.ascontiguousarray(emb_b, np.float32)
        out = np.zeros_like(lm)
        self._ck(self.lib.nhans_masknet(self.h, _ptr(lm), _ptr(fo), len(fo) - 1, _ptr(ea), _ptr(eb), _ptr(out)))
        return out

    def istft(self, logmag, phase, frame_offs, peak=None, want_i16=False):
        lm = np.ascontiguousarray(logmag, np.float32)
        ph = np.ascontiguousarray(phase, np.float32)
        fo = np.ascontiguousarray(frame_offs, np.int64)
        U = len(fo) - 1
        oo = np.zeros(U + 1, np.int64)
        self._ck(self.lib.nhans_istft(self.h, _ptr(lm), _ptr(ph), _ptr(fo), U, None, None, None, _ptr(oo)))
        f32 = np.zeros(int(oo[-1]), np.float32)
        i16 = np.zeros(int(oo[-1]), np.int16) if want_i16 else None
        pk = np.ascontiguousarray(peak, np.int32) if peak is not None else None
        self._ck(self.lib.nhans_istft(self.h, _ptr(lm), _ptr(ph), _ptr(fo), U, _ptr(pk), _ptr(f32), _ptr(i16), _ptr(oo)))
        return (f32, i16, oo) if want_i16 else (f32, oo)

    # ---- fused path ---------------------------------------------------------------------------
    def output_offsets(self, mix_offs):
        oo = np.zeros(len(mix_offs), np.int64)
        rc = self.lib.nhans_output_offsets(_ptr(np.ascontiguousarray(mix_offs, np.int64)), len(mix_offs) - 1, _ptr(oo))
        if rc:
            raise NhansError(rc, "bad offsets")
        return oo

    def enhance_packed(self, mix, mix_offs, ctx_a, a_offs, ctx_b, b_offs, out_i16=None, out_f32=None, mixproc=None, sync=True):
        """Raw (data, offsets) interface used by the benchmark: enqueue H2D + kernels + D2H."""
        U = len(mix_offs) - 1
        self._ck(self.lib.nhans_enhance_batch(self.h, _ptr(mix), _ptr(mix_offs), U, _ptr(ctx_a), _ptr(a_offs), _ptr(ctx_b),
                                              _ptr(b_offs), _ptr(out_i16), _ptr(out_f32), _ptr(mixproc)))
        if sync:
            self.sync()

    # Pinned staging: two sets of grow-only cudaHostAlloc buffers, one per batch the library keeps in flight
    # (nhans_enhance_batch is double buffered), so every H2D / D2H copy is a true asynchronous DMA.
    def _pinned(self, stage, key, n, dtype):
        pool = self.__dict__.setdefault("_stage_bufs", [{}, {}])[stage]
        cur = pool.get(key)
        if cur is None or cur.array.size < n:
            if cur is not None:
                cur.free()
            cur = PinnedArray((max(int(n * 1.25), 1024),), dtype)
            pool[key] = cur
        return cur.array[:n]

    def _pack_pinned(self, stage, key, clips):
        return pack(clips, np.int16, lambda n, dtype: self._pinned(stage, key, n, dtype))

    def submit(self, mix_clips, ctx_a_clips, ctx_b_clips, want_f32=True, want_i16=True, want_mixproc=False):
        """Stage a batch in pinned memory and enqueue H2D + kernels + D2H without waiting.  Up to two batches may be
        in flight: collect() the older one before submitting a third.  -> ticket for collect()."""
        stage = self.__dict__.get("_next_stage", 0)
        busy = self.__dict__.setdefault("_stage_busy", [False, False])
        if busy[stage]:
            raise NhansError(-3, "two batches are already in flight: collect() one first")
        mix, mo = self._pack_pinned(stage, "mix", mix_clips)
        b, bo = self._pack_pinned(stage, "b", ctx_b_clips)
        a, ao = self._pack_pinned(stage, "a", ctx_a_clips) if ctx_a_clips is not None else (None, None)
        oo = self.output_offsets(mo)
        n = int(oo[-1])
        o16 = self._pinned(stage, "o16", n, np.int16) if want_i16 else None
        o32 = self._pinned(stage, "o32", n, np.float32) if want_f32 else None
        mp = self._pinned(stage, "mp", n, np.float32) if want_mixproc else None
        self.enhance_packed(mix, mo, a, ao, b, bo, o16, o32, mp, sync=False)
        busy[stage] = True
        self._next_stage = stage ^ 1
        return dict(stage=stage, oo=oo, o16=o16, o32=o32, mp=mp)

    def collect(self, ticket, newer_in_flight=False):
        """Wait for a submitted batch and copy its outputs out of the staging buffers.  With newer_in_flight the wait
        covers only this (older) batch, so the newer one keeps computing while the caller unpacks."""
        if newer_in_flight:
            self._ck(self.lib.nhans_sync_previous(self.h))
        else:
            self.sync()
        oo = ticket["oo"]
        res = {"out_offs": oo}
        for key, name in (("o16", "i16"), ("o32", "f32"), ("mp", "mixed_processed")):
            if ticket[key] is not None:
                res[name] = [np.array(v) for v in unpack(ticket[key], oo)]      # copies: the staging buffer is reused
        self._stage_busy[ticket["stage"]] = False
        return res

    def enhance(self, mix_clips, ctx_a_clips, ctx_b_clips, want_f32=True, want_i16=True, want_mixproc=False):
        """Lists of int16 clips -> dict of per-utterance outputs.  ctx_a_clips may be None (Silent.wav)."""
        return self.collect(self.submit(mix_clips, ctx_a_clips, ctx_b_clips, want_f32, want_i16, want_mixproc))

    def postmix(self, out_offs, compensate=0.0, ac=False):
        """SN post-mix outputs of the batch just enhanced -> dict of per-utterance lists + snr_est array."""
        n, U = int(out_offs[-1]), len(out_offs) - 1
        mixed, removed, comp = (np.zeros(n, np.float32) for _ in range(3))
        snr = np.zeros(U, np.float32)
        self._ck(self.lib.nhans_postmix(self.h, float(compensate), int(bool(ac)), _ptr(mixed), _ptr(removed), _ptr(comp), _ptr(snr)))
        self.sync()
        return {"mixed_processed": unpack(mixed, out_offs), "removed": unpack(removed, out_offs),
                "compensated": unpack(comp, out_offs), "snr_est": snr}

    # ---- streaming --------------------------------------------------------------------------------
    def stream_open(self, ctx_a_clips, ctx_b_clips, peaks):
        """Open one live int16 stream per context pair (ctx_a_clips may be None: Silent.wav).  peaks: the int16 peak each
        stream is scaled by (the whole clip's nhans_stft peak reproduces the batch path exactly, 32767 is full scale).
        -> list of stream ids"""
        n = len(ctx_b_clips)
        b, bo = pack(ctx_b_clips)
        a, ao = pack(ctx_a_clips) if ctx_a_clips is not None else (None, None)
        pk = np.ascontiguousarray(peaks, np.int32)
        ids = np.zeros(n, np.int32)
        self._ck(self.lib.nhans_stream_open(self.h, n, _ptr(a), _ptr(ao), _ptr(b), _ptr(bo), _ptr(pk), _ptr(ids)))
        return [int(i) for i in ids]

    def stream_step(self, ids, chunks, final=None, want_f32=True, want_i16=True):
        """Append chunks[i] (int16) to stream ids[i] and run every window that became computable; final[i] flushes
        stream i.  -> {"i16": [...], "f32": [...]}: the samples each stream emitted in this step."""
        n = len(ids)
        pcm, offs = pack(chunks)
        ids_a = np.ascontiguousarray(ids, np.int32)
        fin = np.ascontiguousarray(final, np.int32) if final is not None else None
        # a step emits fewer than len(chunk) + 17 * 160 + 400 samples per stream (the frames it held back, plus the last
        # frame's tail at the final step)
        cap = int(offs[-1]) + STREAM_EMIT_SLACK * n
        oo = np.zeros(n + 1, np.int64)
        o16 = np.empty(cap, np.int16) if want_i16 else None
        o32 = np.empty(cap, np.float32) if want_f32 else None
        self._ck(self.lib.nhans_stream_step(self.h, n, _ptr(ids_a), _ptr(pcm), _ptr(offs), _ptr(fin), _ptr(o16), _ptr(o32), _ptr(oo)))
        return {"i16": [np.array(v) for v in unpack(o16, oo)] if want_i16 else None,
                "f32": [np.array(v) for v in unpack(o32, oo)] if want_f32 else None}

    def stream_step_post(self, ids, chunks, compensate, final=None):
        """stream_step plus the post-mix outputs of postmix(compensate, ac=False) for the emitted samples.  compensate: one
        factor for every stream or one per stream.  -> {"i16", "f32", "mixed_processed", "removed", "compensated"}: per-stream
        lists of this step's samples, and "snr_est": each stream's running estimate over its post-step samples so far."""
        n = len(ids)
        pcm, offs = pack(chunks)
        ids_a = np.ascontiguousarray(ids, np.int32)
        fin = np.ascontiguousarray(final, np.int32) if final is not None else None
        comp = np.ascontiguousarray(np.broadcast_to(np.asarray(compensate, np.float32), (n,)))
        cap = int(offs[-1]) + STREAM_EMIT_SLACK * n
        oo = np.zeros(n + 1, np.int64)
        o16 = np.empty(cap, np.int16)
        o32, mixed, removed, compensated = (np.empty(cap, np.float32) for _ in range(4))
        snr = np.zeros(n, np.float32)
        self._ck(self.lib.nhans_stream_step_post(self.h, n, _ptr(ids_a), _ptr(pcm), _ptr(offs), _ptr(fin), _ptr(comp), _ptr(o16),
                                                 _ptr(o32), _ptr(mixed), _ptr(removed), _ptr(compensated), _ptr(oo), _ptr(snr)))
        res = {k: [np.array(v) for v in unpack(a, oo)] for k, a in
               (("i16", o16), ("f32", o32), ("mixed_processed", mixed), ("removed", removed), ("compensated", compensated))}
        res["snr_est"] = snr
        return res

    def stream_close(self, ids):
        ids_a = np.ascontiguousarray(ids, np.int32)
        self._ck(self.lib.nhans_stream_close(self.h, len(ids_a), _ptr(ids_a)))

    def upload(self, mix, mix_offs, ctx_a, a_offs, ctx_b, b_offs):
        self._ck(self.lib.nhans_upload(self.h, _ptr(mix), _ptr(mix_offs), len(mix_offs) - 1, _ptr(ctx_a), _ptr(a_offs),
                                       _ptr(ctx_b), _ptr(b_offs)))

    def run(self):
        self._ck(self.lib.nhans_run(self.h))

    def download(self, out_i16=None, out_f32=None, mixproc=None):
        self._ck(self.lib.nhans_download(self.h, _ptr(out_i16), _ptr(out_f32), _ptr(mixproc)))

    def sync(self):
        self._ck(self.lib.nhans_sync(self.h))

    # ---- measurement / introspection ------------------------------------------------------------
    def event_record(self, slot):
        self._ck(self.lib.nhans_event_record(self.h, slot))

    def event_elapsed_ms(self, a, b):
        ms = ctypes.c_double()
        self._ck(self.lib.nhans_event_elapsed_ms(self.h, a, b, ctypes.byref(ms)))
        return ms.value

    def profile(self, on=True):
        self._ck(self.lib.nhans_profile_enable(self.h, int(on)))

    def profile_reset(self):
        self._ck(self.lib.nhans_profile_reset(self.h))

    def profile_get(self, kind):
        st = np.zeros(4, np.float64)
        self._ck(self.lib.nhans_profile_get(self.h, kind, _ptr(st)))
        return dict(launches=int(st[0]), ms=float(st[1]), flops=float(st[2]), bytes=float(st[3]))

    def profile_layers(self, net=0):
        """Per tensor-core layer: name, launches, ms, algorithmic TFLOP/s."""
        out = []
        for i, g in enumerate(self.plan(net)["gemm"]):
            st = np.zeros(4, np.float64)
            self._ck(self.lib.nhans_profile_get_layer(self.h, net, i, _ptr(st)))
            out.append(dict(name=g["name"], launches=int(st[0]), ms=float(st[1]),
                            tflops=float(st[2] / st[1] / 1e9) if st[1] > 0 else 0.0, K=g["K"], N=g["N"]))
        return out

    def plan(self, net=0):
        return json.loads(self.lib.nhans_plan_json(self.h, net).decode())

    def read_buffer(self, net, buf):
        g = self.plan(net)["bufs"][buf]
        n = g["pixels"] * g["C"]
        out = np.zeros(n, np.uint16)
        self._ck(self.lib.nhans_debug_read_buffer(self.h, net, buf, _ptr(out), n))
        return out.view(np.float16).reshape(g["pixels"], g["C"])

    def read_batch_spectra(self, n_frames):
        """Fused path introspection: (logmag [F,201], unit phasors [F,201,2], denoised logmag [F,201]) of the batch
        just processed, as kept in HBM between the kernels."""
        lm = np.zeros((n_frames, N_BINS), np.float32)
        ph = np.zeros((n_frames, N_BINS, 2), np.float32)
        den = np.zeros((n_frames, N_BINS), np.float32)
        self._ck(self.lib.nhans_debug_read_batch(self.h, 0, _ptr(lm), lm.size))
        self._ck(self.lib.nhans_debug_read_batch(self.h, 1, _ptr(ph), ph.size))
        self._ck(self.lib.nhans_debug_read_batch(self.h, 2, _ptr(den), den.size))
        return lm, ph, den

    def device_info(self):
        sm, ma, mi, mem = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int64()
        self._ck(self.lib.nhans_device_info(self.h, ctypes.byref(sm), ctypes.byref(ma), ctypes.byref(mi), ctypes.byref(mem)))
        return dict(sm_count=sm.value, cc=(ma.value, mi.value), mem_bytes=mem.value)
