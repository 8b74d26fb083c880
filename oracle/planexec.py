"""ctypes wrapper of oracle/_build/libplanexec.so - TEST INFRASTRUCTURE ONLY.

The CPU interpreter of the device layer plan (oracle/plan_exec.cc): same data structures as the CUDA
engine, plain loops.  Used by tests/ to validate nhans_b200/csrc/plan.cc against the oracle without a GPU
and to isolate kernel bugs from plan bugs on the GPU box."""
from __future__ import annotations

import ctypes
import json
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libplanexec.so")


def build():
    subprocess.check_call(["make", "-C", _HERE, "-s"])


def _load():
    if not os.path.exists(_SO):
        build()
    lib = ctypes.CDLL(_SO)
    lib.planexec_create.restype = ctypes.c_void_p
    lib.planexec_error.restype = ctypes.c_char_p
    lib.planexec_plan_json.restype = ctypes.c_char_p
    lib.planexec_plan_json.argtypes = [ctypes.c_void_p, ctypes.c_int]
    lib.planexec_destroy.argtypes = [ctypes.c_void_p]
    return lib


def marshal_weights(weights):
    names = sorted(weights)
    arrs = [np.ascontiguousarray(weights[n], dtype=np.float32) for n in names]
    c_names = (ctypes.c_char_p * len(names))(*[n.encode() for n in names])
    c_sizes = (ctypes.c_int64 * len(names))(*[a.size for a in arrs])
    c_data = (ctypes.c_void_p * len(names))(*[a.ctypes.data for a in arrs])
    return names, arrs, c_names, c_sizes, c_data


class PlanExec:
    def __init__(self, weights, variant=0, win_cap=4, row_cap=1):
        self.lib = _load()
        names, arrs, c_names, c_sizes, c_data = marshal_weights(weights)
        self.h = self.lib.planexec_create(c_names, c_sizes, c_data, len(names), variant, win_cap, row_cap)
        if not self.h:
            raise RuntimeError(self.lib.planexec_error().decode())

    def close(self):
        if self.h:
            self.lib.planexec_destroy(self.h)
            self.h = None

    def plan(self, net=0):
        return json.loads(self.lib.planexec_plan_json(self.h, net).decode())

    def embed(self, ctx_logmag):
        x = np.ascontiguousarray(ctx_logmag, np.float32)
        R = x.shape[0]
        out = np.zeros((R, 512), np.float32)
        self.lib.planexec_embed(ctypes.c_void_p(self.h), x.ctypes.data_as(ctypes.c_void_p), R, out.ctypes.data_as(ctypes.c_void_p))
        return out

    def masknet(self, logmag, frame_offs, emb_a, emb_b):
        lm = np.ascontiguousarray(logmag, np.float32)
        fo = np.ascontiguousarray(frame_offs, np.int64)
        ea = np.ascontiguousarray(emb_a, np.float32)
        eb = np.ascontiguousarray(emb_b, np.float32)
        out = np.zeros_like(lm)
        self.lib.planexec_masknet(ctypes.c_void_p(self.h), lm.ctypes.data_as(ctypes.c_void_p), fo.ctypes.data_as(ctypes.c_void_p),
                                  len(fo) - 1, ea.ctypes.data_as(ctypes.c_void_p), eb.ctypes.data_as(ctypes.c_void_p),
                                  out.ctypes.data_as(ctypes.c_void_p))
        return out

    def cond(self, emb_a, emb_b):
        """Conditioning table of the main network in double -> (cond, cond_abs) [U][cond_cols]."""
        ea = np.ascontiguousarray(emb_a, np.float32)
        eb = np.ascontiguousarray(emb_b, np.float32)
        n_cols = self.plan(0)["cond_cols"]
        cond = np.zeros((ea.shape[0], n_cols))
        cond_abs = np.zeros_like(cond)
        self.lib.planexec_cond(ctypes.c_void_p(self.h), _vp(ea), _vp(eb), ea.shape[0], _vp(cond), _vp(cond_abs))
        return cond, cond_abs

    def first(self, net, units, raw, cond=None):
        """First convolution of `net` in double for a unit table (dict of int arrays frame / lo / hi / utt) ->
        (val, S) [n][Ho][Wo][N]: the value before the fp16 store and the magnitude sum bounding its rounding error."""
        g = self.plan(net)["first"]["out"]
        ut = _units(units)
        n = len(ut[0])
        val = np.zeros((n, g["H"], g["W"], g["C"]))
        S = np.zeros_like(val)
        c, ca = (None, None) if cond is None else (np.ascontiguousarray(cond[0]), np.ascontiguousarray(cond[1]))
        self.lib.planexec_first(ctypes.c_void_p(self.h), net, *[_vp(a) for a in ut], n, _vp(np.ascontiguousarray(raw, np.float32)),
                                _vp(c), _vp(ca), _vp(val), _vp(S))
        return val, S

    def layer(self, net, li, bufs, units, raw, cond=None, errs=None):
        """GemmLayer `li` of `net` evaluated layer-local in double for the units of a unit table (at most this object's
        capacity).  bufs: {buffer index: fp32 [pixels, C] in this object's plan geometry} for every buffer the layer
        reads; errs: the same for bounds of their elements' errors.  -> (val, S, E) [n][Ho][Wo][N] (see plan_exec.cc)."""
        plan = self.plan(net)
        L = plan["gemm"][li]
        ut = _units(units)
        n = len(ut[0])
        nb = len(plan["bufs"])
        arrs = {b: np.ascontiguousarray(a, np.float32) for b, a in bufs.items()}
        earrs = {b: np.ascontiguousarray(a, np.float32) for b, a in (errs or {}).items()}
        c_bufs = (ctypes.c_void_p * nb)(*[arrs[b].ctypes.data if b in arrs else None for b in range(nb)])
        c_errs = (ctypes.c_void_p * nb)(*[earrs[b].ctypes.data if b in earrs else None for b in range(nb)]) if errs else None
        Ho, Wo = (1, 1) if L["out"]["buf"] < 0 else (L["Ho"], L["Wo"])
        val = np.zeros((n, Ho, Wo, L["N"]))
        S = np.zeros_like(val)
        E = np.zeros_like(val)
        c, ca = (None, None) if cond is None else (np.ascontiguousarray(cond[0]), np.ascontiguousarray(cond[1]))
        rc = self.lib.planexec_layer(ctypes.c_void_p(self.h), net, li, c_bufs, c_errs, *[_vp(a) for a in ut], n,
                                     _vp(np.ascontiguousarray(raw, np.float32)), _vp(c), _vp(ca), _vp(val), _vp(S), _vp(E))
        if rc:
            raise RuntimeError(self.lib.planexec_error().decode())
        return val, S, E

    def read_buffer(self, net, buf):
        g = self.plan(net)["bufs"][buf]
        n = g["pixels"] * g["C"]
        out = np.zeros(n, np.float32)
        rc = self.lib.planexec_read_buffer(ctypes.c_void_p(self.h), net, buf, out.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(n))
        if rc:
            raise RuntimeError("no such buffer")
        return out.reshape(g["pixels"], g["C"])


def _vp(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _units(units):
    return [np.ascontiguousarray(units[k], np.int32) for k in ("frame", "lo", "hi", "utt")]


def grid_gather(grid, flat, n_units):
    """Logical [n, H, W, C] view of a padded grid buffer `flat` [pixels, C] (plan.h grid_pixel) for units 0..n_units-1,
    or for the units listed in the array `n_units`."""
    H, W, C = grid["H"], grid["W"], grid["C"]
    n = (np.arange(n_units) if np.isscalar(n_units) else np.asarray(n_units))[:, None, None]
    h = np.arange(H)[None, :, None]
    w = np.arange(W)[None, None, :]
    if grid["mode"] == 1:
        pix = (n * W + w) * H + h
    else:
        y = h + grid["oy"]
        x = w + grid["ox"]
        plane = (y % grid["sh"]) * grid["sw"] + (x % grid["sw"])
        pix = plane * grid["plane_stride"] + n * grid["ustride"] + (y // grid["sh"]) * grid["rstride"] + (x // grid["sw"])
    return flat[pix]


def grid_scatter(grid, logical):
    """Inverse of grid_gather: an fp32 buffer [pixels, C] holding `logical` [n, H, W, C] as units 0..n-1 and zeros
    everywhere else (the padding of every grid is zero)."""
    flat = np.zeros((grid["pixels"], grid["C"]), np.float32)
    pix = grid_gather(grid, np.arange(grid["pixels"])[:, None], logical.shape[0])[..., 0]
    flat[pix] = logical
    return flat
