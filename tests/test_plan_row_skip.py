"""Vertical-padding skip of the tensor-core GEMM layers: a tile of output row ho runs k-group g only if
ho_lo <= ho < ho_hi (plan.h KGroup).  Skipping is exact only if a skipped group reads nothing but zeros, so the marks
are checked here against the padded grid geometry of plan.h (grid_pixel), and the executed MACs against a count
from the layer shapes of SURVEY.md App. B.  No GPU needed."""
import numpy as np
import pytest

from oracle.planexec import PlanExec, grid_gather

# (scope, kh, kw, sh, sw, C): main.py:221-229 (mask network, 35 x 201 window) and :192-197 (towers, 200 x 201 rows)
MAIN = [("resblock1_1", 4, 4, 1, 1, 64), ("resblock1_2", 4, 4, 1, 1, 64), ("resblock2_1", 4, 4, 2, 2, 128),
        ("resblock2_2", 4, 4, 1, 1, 128), ("resblock3_1", 3, 3, 2, 2, 256), ("resblock3_2", 3, 3, 1, 1, 256),
        ("resblock4_1", 3, 3, 2, 2, 512), ("resblock4_2", 3, 3, 1, 1, 512)]
TOWER = [("embedding/noise_resblock1_1", 8, 4, 3, 2, 64), ("embedding/noise_resblock2_1", 8, 4, 3, 2, 128),
         ("embedding/noise_resblock3_1", 4, 4, 1, 1, 256), ("embedding/noise_resblock4_1", 4, 4, 1, 2, 512)]


def _same(n, k, s):
    o = -(-n // s)
    pad = max((o - 1) * s + k - n, 0)
    return o, pad // 2


def _conv_exec_macs(H, W, kh, kw, sh, sw, cin, cout):
    """MACs of a SAME convolution counting only the kernel rows that read inside the image."""
    Ho, pt = _same(H, kh, sh)
    Wo, _ = _same(W, kw, sw)
    live = sum(1 for ho in range(Ho) for i in range(kh) if 0 <= ho * sh + i - pt < H)
    return live * Wo * kw * cin * cout, Ho, Wo


def _expected_exec(blocks, H, W, head):
    """Executed MACs per unit of every GEMM layer, by name, from the shapes alone."""
    out, cin = {}, 1
    for scope, kh, kw, sh, sw, C in blocks:
        m1, Ho, Wo = _conv_exec_macs(H, W, kh, kw, sh, sw, cin, C)
        if cin > 1:                                      # Cin = 1: the first convolution runs on CUDA cores
            out[scope + "_conv1"] = m1
        m2, _, _ = _conv_exec_macs(Ho, Wo, kh, kw, 1, 1, C, C)
        out[scope + "_conv2"] = m2 + (Ho * Wo * cin * C if cin != C else 0)    # + 1x1 transform (rank 1 when Cin = 1)
        H, W, cin = Ho, Wo, C
    if head:
        out["last_conv"] = 26 * 5 * 512 * 512
        out["last_dense"] = 13312 * 201
    return out


def _logical_rows(plan, buf, rowlen, units):
    """Per TMA row of buffer `buf` (rowlen channels each): does it hold a logical pixel of one of `units` units?"""
    g = plan["bufs"][buf]
    pix = np.zeros(g["pixels"], bool)
    pix[grid_gather(g, np.arange(g["pixels"]), units).ravel()] = True
    return pix.reshape(-1, rowlen // g["C"]).any(axis=1)


def _check_marks(plan):
    cap = plan["capacity"]
    for L in plan["gemm"]:
        logical = [_logical_rows(plan, L["a_buf"][a], L["a_rowlen"][a], cap) if L["a_buf"][a] >= 0 else None for a in (0, 1)]
        unit = np.arange(cap)[:, None]
        wo = np.arange(L["Wo"])[None, :]
        assert len(L["group_list"]) == L["groups"]
        for j, g in enumerate(L["group_list"]):
            lo, hi = g["ho"]
            assert 0 <= lo < hi <= L["Ho"], (L["name"], j)
            rows_ok = logical[g["map"]]
            for ho in range(L["Ho"]):
                m = ho * cap * L["Wq"] + unit * L["Wq"] + wo                   # compute rows of output row ho (plan.h)
                reads = False
                for s in g["shift"]:
                    r = (m + g["row_off"] + s).ravel()
                    r = r[(r >= 0) & (r < len(rows_ok))]                           # TMA zero-fills rows outside the tensor
                    reads |= bool(rows_ok[r].any())
                assert reads == (lo <= ho < hi), (L["name"], j, ho, g)
        # the kernel runs, per output row, the groups [s0, e0) and then [s1, e1): exactly the live ones, in order
        assert len(L["row_groups"]) == L["Ho"]
        for ho, (s0, e0, s1, e1) in enumerate(L["row_groups"]):
            live = [j for j, g in enumerate(L["group_list"]) if g["ho"][0] <= ho < g["ho"][1]]
            assert live and list(range(s0, e0)) + list(range(s1, e1)) == live, (L["name"], ho)


@pytest.mark.parametrize("variant", [0, 1])
def test_dead_groups_match_grid_geometry(variant, weights_sn, weights_ss):
    w = weights_sn if variant == 0 else weights_ss
    ranges = {}
    for win_cap, row_cap in ((1, 1), (3, 2)):
        pe = PlanExec(w, variant, win_cap=win_cap, row_cap=row_cap)
        for net in (0, 1):
            plan = pe.plan(net)
            _check_marks(plan)
            ranges.setdefault(net, []).append({L["name"]: [tuple(g["ho"]) for g in L["group_list"]] for L in plan["gemm"]})
            # the skip is not vacuous: every layer with a kernel taller than 1 has groups that some rows skip
            for L in plan["gemm"]:
                if L["name"] not in ("last_conv", "last_dense"):
                    assert any(tuple(g["ho"]) != (0, L["Ho"]) for g in L["group_list"]), L["name"]
        pe.close()
    for a, b in ranges.values():
        assert a == b, "group row ranges depend on the capacity"


@pytest.mark.parametrize("variant", [0, 1])
def test_executed_macs_match_shapes(variant, weights_sn, weights_ss):
    w = weights_sn if variant == 0 else weights_ss
    pe = PlanExec(w, variant, win_cap=2, row_cap=1)
    for net, blocks, H, head in ((0, MAIN, 35, True), (1, TOWER, 200, False)):
        plan = pe.plan(net)
        want = _expected_exec(blocks, H, 201, head)
        got = {L["name"]: L["exec_macs"] for L in plan["gemm"]}
        assert sorted(got) == sorted(want)
        for name, v in want.items():
            assert got[name] == pytest.approx(v, rel=1e-12, abs=0.5), name
        for L in plan["gemm"]:
            assert L["exec_macs"] <= L["macs"]
        # stage 4 of the mask network: 2 of 15 (output row, kernel row) pairs are padding
        if net == 0:
            L = next(L for L in plan["gemm"] if L["name"] == "resblock4_2_conv1")
            assert L["exec_macs"] == pytest.approx(L["macs"] * 13 / 15, rel=1e-12)
    pe.close()
