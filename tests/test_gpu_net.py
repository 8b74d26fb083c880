"""tcgen05 network kernels through the C ABI: tight against the CPU plan interpreter (same fp16 data
path), and within the stated tolerance against the fp32 oracle."""
import numpy as np
import pytest
import torch

from nhans_b200 import synth
from oracle import nhans_oracle as O
from oracle.planexec import PlanExec, grid_gather

pytestmark = pytest.mark.gpu

REL_TOL = 1e-3            # relative (Frobenius) error of embeddings / mask vs the fp32 oracle
EXEC_TOL = 2e-4           # vs the CPU interpreter of the same fp16 plan (accumulation order only)


def _rel(a, b):
    return float(np.linalg.norm(a.astype(np.float64) - b) / (np.linalg.norm(b) + 1e-30))


def test_embedding_tower(engine_sn, weights_sn, oracle_sn):
    ctx = np.stack([O.context_of(O.logmag_phase(O.normalise(synth.noise_clip(u)))[0]) for u in range(6)])   # > row capacity 4
    emb = engine_sn.embed(ctx)
    with torch.no_grad():
        ref = oracle_sn.tower(torch.from_numpy(ctx)).numpy()
    assert _rel(emb, ref) < REL_TOL
    pe = PlanExec(weights_sn, 0, win_cap=1, row_cap=1)
    assert _rel(emb[:2], pe.embed(ctx[:2])) < EXEC_TOL
    pe.close()
    sil = np.full((1, 200, 201), np.log(np.float32(1e-5)), np.float32)                                       # Silent.wav context
    with torch.no_grad():
        ref = oracle_sn.tower(torch.from_numpy(sil)).numpy()
    assert _rel(engine_sn.embed(sil), ref) < REL_TOL


@pytest.mark.parametrize("variant", [0, 1])
def test_masknet_layers_and_output(variant, engine_sn, engine_ss, weights_sn, weights_ss, oracle_sn, oracle_ss, monkeypatch):
    eng = engine_sn if variant == 0 else engine_ss
    w = weights_sn if variant == 0 else weights_ss
    net = oracle_sn if variant == 0 else oracle_ss
    mixes = [synth.mixture(0.2, 0)[:400 + 160 * 5], synth.mixture(0.2, 1)[:400 + 160 * 2]]      # 6 + 3 windows
    lms = [O.logmag_phase(O.normalise(m))[0] for m in mixes]
    fo = np.cumsum([0] + [l.shape[0] for l in lms])
    lm = np.concatenate(lms)
    rng = np.random.default_rng(variant)
    ea = rng.normal(0, 2, (2, 512)).astype(np.float32)
    eb = rng.normal(0, 2, (2, 512)).astype(np.float32)
    den = eng.masknet(lm, fo, ea, eb)
    pe = PlanExec(w, variant, win_cap=256, row_cap=1)
    den_pe = pe.masknet(lm, fo, ea, eb)
    assert _rel(den - lm, den_pe - lm) < 2e-3 and np.abs(den - den_pe).max() < 2e-3
    plan = eng.plan(0)
    assert plan["bufs"] == pe.plan(0)["bufs"]
    first_buf = plan["first"]["out"]["buf"]
    # (every tensor-core layer's grid is checked elementwise, layer-local, in test_gpu_net_flavours.py)
    # the first convolution's output is not materialised by this engine: resblock1_1_conv2 builds its operand from the
    # per-frame table (conv_walk.cu kWalkGen).  The same engine path with the operand generator switched off stores it
    monkeypatch.setenv("NHANS_NO_GEN", "1")
    from nhans_b200.engine import Engine
    nogen = Engine(0, variant, win_capacity=256, row_capacity=4)
    try:
        nogen.load_weights(w)
        den2 = nogen.masknet(lm, fo, ea, eb)
        g = plan["bufs"][first_buf]
        a = grid_gather(g, nogen.read_buffer(0, first_buf).astype(np.float32), 9)
        assert a.any() and _rel(a, grid_gather(g, pe.read_buffer(0, first_buf), 9)) < 1e-3
        assert np.abs(den2 - den).max() < 2e-3               # generated operand == materialised operand (fp16 rounding of the same values)
    finally:
        nogen.close()
    pe.close()
    ref = []
    with torch.no_grad():
        for u, l in enumerate(lms):
            win = torch.from_numpy(O.strided_crop(l, 35))
            T = win.shape[0]
            ref.append(net.mask_net(win, torch.from_numpy(ea[u:u + 1]).expand(T, -1), torch.from_numpy(eb[u:u + 1]).expand(T, -1)).numpy())
    ref = np.concatenate(ref)
    # mask = exp(out): relative mask error == absolute error of out
    assert _rel(np.exp(den - lm), np.exp(ref - lm)) < REL_TOL
    assert _rel(den - lm, ref - lm) < 2e-3


def test_padding_positions_stay_zero(engine_sn):
    """The grids' padding slots implement the conv zero padding; no kernel may ever write them."""
    rng = np.random.default_rng(5)
    lm = rng.normal(-3, 2, (300, 201)).astype(np.float32)     # > win capacity 256 -> 2 passes
    engine_sn.masknet(lm, np.array([0, 120, 300]), rng.normal(0, 1, (2, 512)).astype(np.float32), rng.normal(0, 1, (2, 512)).astype(np.float32))
    plan = engine_sn.plan(0)
    for g in plan["bufs"]:
        if g["mode"] != 0:
            continue
        buf = engine_sn.read_buffer(0, g["buf"])
        mask = np.ones(g["pixels"], bool)
        pix = grid_gather(g, np.arange(g["pixels"])[:, None], plan["capacity"])[..., 0]
        mask[pix.ravel()] = False
        assert not np.any(buf[mask]), g


def test_row_walk_matches_plain_gemm(engine_sn, weights_sn, monkeypatch):
    """The 64-channel stage runs on the row-walk kernel (conv_walk.cu); NHANS_NO_WALK=1 executes the same layers as
    plain N = 64 shifted-row GEMMs.  Same fp16 operands, same fp32 products, other summation order: every activation
    grid of the stage agrees to fp16 rounding noise, over several passes and a ragged last tile."""
    from nhans_b200.engine import Engine
    rng = np.random.default_rng(11)
    lm = rng.normal(-3, 2, (300 + 77, 201)).astype(np.float32)         # 256 + 121 windows: 2 passes, 3 utterances
    fo = np.array([0, 40, 300, 377])
    ea = rng.normal(0, 1, (3, 512)).astype(np.float32)
    eb = rng.normal(0, 1, (3, 512)).astype(np.float32)
    assert sum(g["walk"] for g in engine_sn.plan(0)["gemm"]) == 3
    den = engine_sn.masknet(lm, fo, ea, eb)
    monkeypatch.setenv("NHANS_NO_WALK", "1")
    monkeypatch.setenv("NHANS_NO_SPLITK", "1")                        # and last_dense as one K loop instead of 8 splits + reduce
    plain = Engine(0, 0, win_capacity=256, row_capacity=4)
    try:
        plain.load_weights(weights_sn)
        den_p = plain.masknet(lm, fo, ea, eb)
        assert np.abs(den - den_p).max() < 2e-3
        assert np.isfinite(den).all()                                  # (the first pass, 256 windows, takes the split-K head)
        for g in engine_sn.plan(0)["gemm"]:
            if not g["walk"]:
                continue
            grid = g["out"]
            a = grid_gather(grid, engine_sn.read_buffer(0, grid["buf"]).astype(np.float32), 121)
            b = grid_gather(grid, plain.read_buffer(0, grid["buf"]).astype(np.float32), 121)
            assert _rel(a, b) < 2e-4, g["name"]
            assert np.abs(a - b).max() <= 2e-3 * max(1.0, float(np.abs(b).max())), g["name"]
    finally:
        plain.close()
