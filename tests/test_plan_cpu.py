"""The device layer plan (nhans_b200/csrc/plan.cc: grids, k-block offsets, weight packing, BN / embedding
folding) interpreted on the CPU must reproduce the oracle network - proves the plan without a GPU."""
import numpy as np
import pytest
import torch

from nhans_b200 import synth
from oracle import nhans_oracle as O
from oracle.planexec import PlanExec, grid_gather


def _rel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def test_tower_plan_matches_oracle(weights_sn, oracle_sn):
    pe = PlanExec(weights_sn, 0, win_cap=2, row_cap=1)
    ctx = np.stack([O.context_of(O.logmag_phase(O.normalise(synth.noise_clip(u)))[0]) for u in range(2)])
    emb = pe.embed(ctx)                                    # two passes of capacity 1
    with torch.no_grad():
        ref = oracle_sn.tower(torch.from_numpy(ctx)).numpy()
    assert _rel(emb, ref) < 1e-3                           # fp16 operands, fp32 accumulation
    plan = pe.plan(1)
    assert [g["name"] for g in plan["gemm"]][-1] == "embedding/noise_resblock4_1_conv2"
    assert abs(sum(g["macs"] for g in plan["gemm"]) + plan["first"]["macs"] - 7557428160) < 1    # SURVEY App. B
    pe.close()


@pytest.mark.parametrize("variant", [0, 1])
def test_masknet_plan_matches_oracle(variant, weights_sn, weights_ss, oracle_sn, oracle_ss):
    w = weights_sn if variant == 0 else weights_ss
    net = oracle_sn if variant == 0 else oracle_ss
    pe = PlanExec(w, variant, win_cap=3, row_cap=1)
    plan = pe.plan(0)
    assert abs(sum(g["macs"] for g in plan["gemm"]) + plan["first"]["macs"] - 5163572928) < 1      # 10.327 GFLOP / window
    mixes = [synth.mixture(0.07, 0)[:400 + 160 * 3], synth.mixture(0.06, 1)[:400 + 160 * 1]]      # 4 + 2 windows, chunks of 3
    lms = [O.logmag_phase(O.normalise(m))[0] for m in mixes]
    fo = np.cumsum([0] + [l.shape[0] for l in lms])
    lm = np.concatenate(lms)
    rng = np.random.default_rng(0)
    ea = rng.normal(0, 2, (2, 512)).astype(np.float32)
    eb = rng.normal(0, 2, (2, 512)).astype(np.float32)
    den = pe.masknet(lm, fo, ea, eb)
    ref, taps = [], {}
    with torch.no_grad():
        for u, l in enumerate(lms):
            win = torch.from_numpy(O.strided_crop(l, 35))
            T = win.shape[0]
            taps = {}
            ref.append(net.mask_net(win, torch.from_numpy(ea[u:u + 1]).expand(T, -1), torch.from_numpy(eb[u:u + 1]).expand(T, -1), taps).numpy())
    ref = np.concatenate(ref)
    assert _rel(den - lm, ref - lm) < 2e-3                 # mask (= exp(out)) within ~1e-3 relative
    assert np.abs(den - ref).max() < 5e-3
    # last chunk = utterance 1's windows [1:2] -> unit 0..: compare block outputs stored in the padded grids
    names = {n: next(g["out"]["buf"] for g in plan["gemm"] if g["name"] == n + "_conv2")
             for n in ("resblock1_1", "resblock2_2", "resblock4_1")}
    n_last = int(fo[-1]) - 3
    first_unit_global = 3                                  # chunk 2 starts at global window 3 = utt 1, window 0... (4 windows in utt 0)
    for name, buf in names.items():
        g = plan["bufs"][buf]
        got = grid_gather(g, pe.read_buffer(0, buf), n_last)
        want = taps[name].numpy()                          # taps of the last utterance (2 windows)
        # chunk 2 holds global windows 3,4,5 = (utt0 w3), (utt1 w0), (utt1 w1)
        assert _rel(got[1:3], want) < 2e-3, name
    pe.close()


def test_plan_geometry_invariants(weights_sn):
    pe = PlanExec(weights_sn, 0, win_cap=2, row_cap=1)
    for net in (0, 1):
        plan = pe.plan(net)
        for g in plan["gemm"]:
            assert g["K"] % 64 == 0 and g["N"] % 16 == 0 and g["N"] % g["BN"] == 0 and g["BN"] <= 256
        for b in plan["bufs"]:
            if b["mode"] == 0:
                # every logical pixel maps to a distinct in-range slot
                n = 2 if net == 0 else 1
                pix = grid_gather(b, np.arange(b["pixels"])[:, None], n)[..., 0]
                assert pix.min() >= 0 and pix.max() < b["pixels"] and len(np.unique(pix)) == pix.size
    pe.close()


def test_tiny_last_dense_keeps_precision(weights_sn):
    """last_dense is zero-initialised in the reference and trained with lr 1e-3, so a real checkpoint may hold
    weights around 1e-5 - below the fp16 normal range (6.1e-5).  The plan scales every output column by a power of
    two before the fp16 cast and undoes it in the head epilogue, so the mask keeps its relative accuracy."""
    w = dict(weights_sn)
    w["last_dense/w"] = (w["last_dense/w"] * np.float32(1e-5 / np.abs(w["last_dense/w"]).max())).astype(np.float32)
    w["last_dense/b"] = (w["last_dense/b"] * np.float32(1e-2)).astype(np.float32)
    assert np.abs(w["last_dense/w"]).max() < 2e-5
    pe = PlanExec(w, 0, win_cap=4, row_cap=1)
    net = O.Net(w, 0)
    lm = O.logmag_phase(O.normalise(synth.mixture(0.07, 4)[:400 + 160 * 3]))[0]            # 4 windows
    rng = np.random.default_rng(3)
    ea = rng.normal(0, 2, (1, 512)).astype(np.float32)
    eb = rng.normal(0, 2, (1, 512)).astype(np.float32)
    den = pe.masknet(lm, np.array([0, lm.shape[0]]), ea, eb)
    with torch.no_grad():
        win = torch.from_numpy(O.strided_crop(lm, 35))
        ref = net.mask_net(win, torch.from_numpy(ea).expand(4, -1), torch.from_numpy(eb).expand(4, -1)).numpy()
    assert np.abs(ref - lm).max() > 0                       # the head still contributes
    assert _rel(den - lm, ref - lm) < 2e-3                  # a plain fp16 cast of 1e-5 weights loses ~2 decimal digits
    pe.close()


def _pass_units(fo, w0, n):
    """Unit table of windows w0 .. w0 + n - 1 (one window per frame) of utterances with frame offsets fo."""
    g = np.arange(w0, w0 + n)
    utt = np.searchsorted(fo, g, side="right") - 1
    return dict(frame=g, lo=fo[utt], hi=fo[utt + 1], utt=utt)


def test_layer_evaluator_matches_interpreter(weights_sn):
    """The layer-local double evaluator (planexec_layer / planexec_first), fed the interpreter's own grids, agrees with
    the interpreter's fp32 run elementwise within the accumulation bound of tests/layercheck.py, for every layer, unit
    and pixel of the last pass of both networks, den and the pooled embedding included; and again from grids
    compacted to a subset of the units at another capacity (how the GPU tests feed it)."""
    import layercheck as LC
    rng = np.random.default_rng(7)
    fo = np.array([0, 3, 5, 7])                                  # 3 utterances, 7 windows: passes of 4 + 3
    lm = rng.normal(-3, 2, (7, 201)).astype(np.float32)
    ea = rng.normal(0, 2, (3, 512)).astype(np.float32)
    eb = rng.normal(0, 2, (3, 512)).astype(np.float32)
    pe = PlanExec(weights_sn, 0, win_cap=4, row_cap=2)
    small = PlanExec(weights_sn, 0, win_cap=2, row_cap=1)
    try:
        den = pe.masknet(lm, fo, ea, eb)
        plan = pe.plan(0)
        ut = _pass_units(fo, 4, 3)
        cond = pe.cond(ea, eb)
        read = lambda b: pe.read_buffer(0, b)
        v, S = pe.first(0, ut, lm, cond)
        got = grid_gather(plan["first"]["out"], read(plan["first"]["out"]["buf"]), 3)
        assert LC.compare("first", got, v, LC.ulp16(v) + LC.C_ACC * S, str) <= 1.0
        every = {li: range(3) for li in range(len(plan["gemm"]))}
        r = LC.check_pass(pe, 0, plan, read, ut, every, lm, cond, den=den[4:])
        assert len(r) == len(plan["gemm"]) and max(r.values()) <= 1.0
        r2 = LC.check_pass(small, 0, plan, read, ut, {li: [0, 2] for li in every}, lm, cond, den=den[4:], gen_first=True)
        assert max(r2.values()) <= 1.0

        ctx = np.stack([O.context_of(O.logmag_phase(O.normalise(synth.noise_clip(u)))[0]) for u in range(3)])
        emb = pe.embed(ctx)                                      # passes of 2 + 1 context rows
        tplan = pe.plan(1)
        raw = ctx.reshape(-1, 201)
        tut = dict(frame=[400], lo=[400], hi=[600], utt=[0])
        tread = lambda b: pe.read_buffer(1, b)
        v, S = pe.first(1, tut, raw)
        got = grid_gather(tplan["first"]["out"], tread(tplan["first"]["out"]["buf"]), 1)
        assert LC.compare("tower first", got, v, LC.ulp16(v) + LC.C_ACC * S, str) <= 1.0
        r = LC.check_pass(small, 1, tplan, tread, tut, {li: [0] for li in range(len(tplan["gemm"]))}, raw)
        assert max(r.values()) <= 1.0
        pool = grid_gather(tplan["bufs"][tplan["pool_buf"]], tread(tplan["pool_buf"]), 1).astype(np.float64).reshape(-1, 512)
        assert np.all(np.abs(emb[2] - pool.mean(0)) <= LC.C_ACC * np.abs(pool).mean(0) + 2.0 ** -23 * np.abs(pool.mean(0)))
    finally:
        pe.close()
        small.close()
