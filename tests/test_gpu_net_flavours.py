"""Every tensor-core layer of both networks, elementwise against the layer-local double evaluator (tests/layercheck.py),
at the pass sizes that switch its kernel path.  Which path a layer takes depends on the units (windows or context rows)
in the pass, M = units * Ho * Wq output rows, and the SM count n_sm (gemm_tc.cu launch_gemm, conv_walk.cu launch_walk):

* CTA pairs when BN % 32 == 0, the layer is not the head and M >= 256 * (n_sm / 2);
* a tile is mt * 128 << cta2 plane rows (mt = 256 / BN, at least 1); the second CTA of the last pair holds part of
  the plane's last rows, or none of them when the plane ends in the first 128 rows of the last 256-row sub-tile;
* the row-walk layers give a CTA more than one 128-row tile when ceil(units * Wq / 128) > n_sm;
* last_dense runs split-K with a partial last 128-unit tile whenever units % 128 != 0.

On 148 SMs the mask network's layers switch to CTA pairs at 11 (resblock2), 41 (resblock3), 141 (resblock4) and 729
(last_conv) windows, the walk layers (Wq = 203) go multi-tile from 94 windows, and the tower's layers switch at 3
(64 channels), 16 (resblock2/3) and 30 (resblock4) rows.  An empty second CTA needs the last tile to end within 128
rows of its start: resblock2 (Wq = 103, 512-row tiles) at 11 and 40 windows, resblock3 (Wq = 52) at 41 and 729,
resblock4 (Wq = 27) first at 143, last_conv (Wq = 26) at 729 (a partial one at 734); in the tower at 16, 29, 30 and
32 rows.  test_pass_sizes_cover_every_path recomputes all of this from the plan and the device's n_sm, so a change of
the selection rule fails there instead of silently losing coverage.

Each size is its own call (only a call's last pass survives in the buffers), over several utterances of uneven length
so that tiles span an utterance boundary.  Per call and layer at most 48 (mostly 10 to 20) units are checked: the pass's first and last
unit, the units on either side of the last two tile boundaries and of every 128-row sub-tile / CTA half inside them,
each utterance's first and last window, and two seeded random ones."""
import numpy as np
import pytest

import layercheck as LC
from oracle.planexec import PlanExec, grid_gather

pytestmark = pytest.mark.gpu

MASK_SIZES = [9, 10, 11, 40, 41, 140, 141, 143, 728, 729]  # variant-0 engine of capacity 768
FULL_SIZE = 2048                                           # one full pass of the default capacity
SS_SIZE = 734                                              # the separator weights (variant 1), same layer geometry
TOWER_SIZES = [2, 3, 15, 16, 29, 30, 32, 33]               # row capacity 32: 33 = passes of 32 + 1
MAX_UNITS = 48


@pytest.fixture(scope="module")
def eng768(weights_sn):
    from nhans_b200.engine import Engine
    e = Engine(0, 0, win_capacity=768, row_capacity=32)
    e.load_weights(weights_sn)
    yield e
    e.close()


@pytest.fixture(scope="module")
def n_sm(eng768):
    return eng768.device_info()["sm_count"]


@pytest.fixture(scope="module")
def evaluators(weights_sn, weights_ss):
    pes = {v: PlanExec(w, v, win_cap=MAX_UNITS, row_cap=MAX_UNITS) for v, w in ((0, weights_sn), (1, weights_ss))}
    yield pes
    for pe in pes.values():
        pe.close()


def _lengths(n, parts):
    """n split into uneven positive parts (one window per frame)."""
    cut = np.unique(np.clip(np.round(np.cumsum(parts)[:-1] * n / sum(parts)).astype(int), 1, n - 1)) if n > 1 else []
    return np.diff(np.concatenate([[0], cut, [n]])).astype(np.int64)


def _select(L, units, n_sm, edges, rng):
    """Units of one layer to check (see the module docstring)."""
    must = {0, units - 1} | LC.boundary_units(L, units, n_sm) | set(edges)
    must = sorted(u for u in must if 0 <= u < units)
    if len(must) > MAX_UNITS:                                 # keep both ends and an even spread of the rest
        must = sorted(set(must[:4] + must[-4:] + must[4:-4:max(1, (len(must) - 8) // (MAX_UNITS - 8) + 1)]))[:MAX_UNITS]
    extra = [u for u in rng.permutation(units) if u not in must][:max(0, min(2, MAX_UNITS - len(must)))]
    return sorted(must + [int(u) for u in extra])


def _run_masknet(eng, pe, n, n_sm, seed):
    rng = np.random.default_rng(seed)
    lens = _lengths(n, [5, 1, 3])
    fo = np.concatenate([[0], np.cumsum(lens)])
    U = len(lens)
    lm = rng.normal(-3, 2, (n, 201)).astype(np.float32)
    ea = rng.normal(0, 2, (U, 512)).astype(np.float32)
    eb = rng.normal(0, 2, (U, 512)).astype(np.float32)
    den = eng.masknet(lm, fo, ea, eb)
    plan = eng.plan(0)
    g = np.arange(n)
    utt = np.searchsorted(fo, g, side="right") - 1
    ut = dict(frame=g, lo=fo[utt], hi=fo[utt + 1], utt=utt)
    edges = list(fo[:-1]) + list(fo[1:] - 1)
    sel = {li: _select(L, n, n_sm, edges, rng) for li, L in enumerate(plan["gemm"])}
    # layer 0's operand is generated from the first convolution's per-frame table and never stored
    return LC.check_pass(pe, 0, plan, lambda b: eng.read_buffer(0, b), ut, sel, lm, pe.cond(ea, eb), den=den, gen_first=True,
                         n_sm=n_sm)


def _report(tag, ratios):
    print("\n%s max |gpu - ref| / bound: %s" % (tag, " ".join("%s=%.3f" % (k.split("/")[-1], v) for k, v in ratios.items())))


def _path(L, n, n_sm):
    cta2, rows, tiles = LC.gemm_path(L, n, n_sm)
    if L["walk"]:
        return "multi-tile" if tiles > n_sm else "one tile"
    if not cta2:
        return "single"
    tail = n * L["Wq"] - (tiles - 1) * rows                 # plane rows of the last tile
    return "pair-empty" if tail <= 128 else "pair-partial" if tail < rows else "pair-full"


def test_pass_sizes_cover_every_path(eng768, evaluators, n_sm):
    """Across the sizes below every layer runs every path that some pass size up to the capacity gives it: single-CTA,
    CTA pairs with a partial second CTA, CTA pairs with an empty second CTA, and for the walk layers one and more than one
    tile per CTA (a pair whose last tile is full is not needed: nothing in it is ragged).  The head runs a partial last
    128-unit tile."""
    geometry = lambda plan: [(L["Wq"], L["Ho"], L["BN"], L["walk"]) for L in plan["gemm"]]
    assert geometry(evaluators[1].plan(0)) == geometry(eng768.plan(0))
    for net, sizes, cap in ((0, MASK_SIZES + [SS_SIZE, FULL_SIZE], FULL_SIZE), (1, [(R - 1) % 32 + 1 for R in TOWER_SIZES], 32)):
        for L in eng768.plan(net)["gemm"]:
            seen = {_path(L, n, n_sm) for n in sizes}
            want = {_path(L, n, n_sm) for n in range(1, cap + 1)} - {"pair-full"}
            assert want <= seen, (net, L["name"], sorted(want - seen))
            if L["out"]["buf"] < 0:
                assert any(n % 128 for n in sizes)


@pytest.mark.parametrize("n", MASK_SIZES)
def test_masknet_layers(n, eng768, evaluators, n_sm):
    _report("masknet %d windows:" % n, _run_masknet(eng768, evaluators[0], n, n_sm, n))


def test_masknet_layers_full_pass(weights_sn, evaluators, n_sm):
    from nhans_b200.engine import Engine
    eng = Engine(0, 0, row_capacity=32)
    try:
        eng.load_weights(weights_sn)
        assert eng.plan(0)["capacity"] == FULL_SIZE
        _report("masknet %d windows:" % FULL_SIZE, _run_masknet(eng, evaluators[0], FULL_SIZE, n_sm, 1))
    finally:
        eng.close()


def test_masknet_layers_separator(weights_ss, evaluators, n_sm):
    from nhans_b200.engine import Engine
    eng = Engine(0, 1, win_capacity=768, row_capacity=32)
    try:
        eng.load_weights(weights_ss)
        _report("separator %d windows:" % SS_SIZE, _run_masknet(eng, evaluators[1], SS_SIZE, n_sm, 2))
    finally:
        eng.close()


@pytest.mark.parametrize("R", TOWER_SIZES)
def test_tower_layers_and_pool(R, eng768, evaluators, n_sm):
    pe = evaluators[0]
    rng = np.random.default_rng(100 + R)
    ctx = rng.normal(-3, 2, (R, 200, 201)).astype(np.float32)
    emb = eng768.embed(ctx)
    plan = eng768.plan(1)
    cap = plan["capacity"]
    r0 = (R - 1) // cap * cap
    n = R - r0
    rows = np.arange(r0, R)
    ut = dict(frame=rows * 200, lo=rows * 200, hi=rows * 200 + 200, utt=np.zeros(n, np.int64))
    sel = {li: _select(L, n, n_sm, [], rng) for li, L in enumerate(plan["gemm"])}
    read = lambda b: eng768.read_buffer(1, b)
    raw = ctx.reshape(-1, 201)
    units = np.array(sel[0])
    v, S = pe.first(1, {k: a[units] for k, a in ut.items()}, raw)
    got = grid_gather(plan["first"]["out"], read(plan["first"]["out"]["buf"]), units)
    ratios = {"first": LC.compare("tower first", got, v, LC.ulp16(v) + LC.C_ACC * S, lambda u, wo: str(units[u]))}
    ratios.update(LC.check_pass(pe, 1, plan, read, ut, sel, raw, n_sm=n_sm))
    # mean_pool_kernel: fp32 mean of the last pass's pool grid
    pool = grid_gather(plan["bufs"][plan["pool_buf"]], read(plan["pool_buf"]), n).astype(np.float64).reshape(n, -1, 512)
    ref = pool.mean(1)
    bound = LC.C_ACC * np.abs(pool).mean(1) + 2.0 ** -23 * np.abs(ref)
    ratios["pool"] = float(np.max(np.abs(emb[r0:] - ref) / np.maximum(bound, 1e-30)))
    _report("tower %d rows:" % R, ratios)
    assert ratios["pool"] <= 1.0
