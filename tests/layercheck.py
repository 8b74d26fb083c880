"""Layer-local check of one pass of a network against the double evaluator of oracle/plan_exec.cc (planexec_layer).

Every tensor-core layer is evaluated from the very inputs the checked implementation read (its own input grids, read
back after the pass), so a layer is judged on its own arithmetic and an error cannot hide behind, or be blamed on, an
earlier layer.  Each value is compared elementwise:

    |got - ref| <= ulp16(ref) + C_ACC * S + E

* ulp16(ref): the fp16 rounding of the stored output (at most half an fp16 ulp of the stored value; one ulp of the
  reference covers it); dropped for the fp32 head output den.
* S = sum |a w| over the K products plus the magnitudes of the epilogue terms (bias or conditioning sum, embedding
  tables, residual, rank-1 raw term, the head's raw row).  An fp32 sum of K terms in any order and grouping is within
  K * u * sum |terms| of the exact sum, with u = 2^-23 the relative error of one fp32 add that rounds or truncates to a
  neighbour (2^-24 for round-to-nearest).  With the largest K of either network, K = 13312 (last_dense), that is
  C_ACC = 13312 * 2^-23 = 1.59e-3 for every layer; the epilogue adds fewer than 8 more fp32 operations, and its fp16
  copies of the time / frequency tables (2^-11 relative) are counted in S through their magnitudes.
* E = sum |w| err(a): only where an input is not the checked implementation's own (layer 0 of the mask network, whose
  operand the engine generates on the fly from the first convolution and never stores; see check_pass).
"""
import numpy as np

from oracle.planexec import grid_gather, grid_scatter

C_ACC = 13312 * 2.0 ** -23


def ulp16(x):
    return np.spacing(np.abs(x).astype(np.float16)).astype(np.float64)


def gemm_path(L, units, n_sm):
    """(cta2, tile rows, tiles per output row) of a layer's launch for a pass of `units` units (api.cu run_net,
    gemm_tc.cu launch_gemm, conv_walk.cu launch_walk)."""
    plane_rows = units * L["Wq"]
    head = L["out"]["buf"] < 0
    if L["walk"]:
        return False, 128, -(-plane_rows // 128)
    cta2 = L["BN"] % 32 == 0 and not head and units * L["Ho"] * L["Wq"] >= 256 * (n_sm // 2)
    rows = (max(1, 256 // L["BN"]) * 128) << int(cta2)
    return cta2, rows, -(-plane_rows // rows)


def boundary_units(L, units, n_sm):
    """Units owning the plane rows on either side of the last two tile boundaries and of every 128-row sub-tile / CTA
    half inside the last two tiles; for a walk layer also of the first tile a CTA takes after its first one."""
    _, rows, tiles = gemm_path(L, units, n_sm)
    plane_rows = units * L["Wq"]
    out = set()
    if L["walk"] and tiles > n_sm:
        out.update(u for u in ((n_sm * rows - 1) // L["Wq"], n_sm * rows // L["Wq"]) if u < units)
    for t in range(max(0, tiles - 2), tiles):
        for r in range(t * rows, min((t + 1) * rows, plane_rows), 128):
            out.update(u for u in ((r - 1) // L["Wq"], r // L["Wq"]) if 0 <= u < units)
    return out


def where(L, units, n_sm, unit, wo):
    """Tile / CTA rank of a unit's output row, for failure messages."""
    cta2, rows, _ = gemm_path(L, units, n_sm)
    r = unit * L["Wq"] + wo
    return "tile %d of %d rows, CTA rank %d" % (r // rows, rows, (r % 256) // 128 if cta2 else 0)


def compare(name, got, ref, bound, ctx):
    """Max ratio |got - ref| / bound; raises with the location of the worst element when it exceeds 1.
    got / ref / bound [n][Ho][Wo][C]; ctx(unit index, wo) -> text."""
    ratio = np.abs(got.astype(np.float64) - ref) / bound
    i = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
    worst = float(ratio[i])
    if not worst <= 1.0:
        u, ho, wo, c = i
        raise AssertionError("%s: unit %s ho %d wo %d channel %d: got %r ref %r bound %.3g (ratio %.3g), %s; %d elements over"
                             % (name, ctx(u, None), ho, wo, c, float(got[i]), float(ref[i]), float(bound[i]), worst,
                                ctx(u, wo), int(np.sum(ratio > 1.0))))
    return worst


def check_pass(pe, net, plan, read, ut, sel, raw, cond=None, den=None, gen_first=False, n_sm=148):
    """Checks every layer of one pass of network `net` (0: mask network, 1: embedding tower).

    plan / read(b): the checked implementation's plan JSON and buffer b as [pixels, C] (only its last pass survives);
    ut: unit table of that pass (dict of int arrays frame / lo / hi / utt); sel: {layer index: unit indices to check}
    (each at most pe's capacity); pe: the evaluator, built for the same weights; raw: fp32 rows the unit table indexes;
    cond: (cond, cond_abs) of the pass's utterances; den: the head's output rows of the pass; gen_first: layer 0's input
    grid was never stored, take it from the evaluator's first convolution.  -> {layer name: max ratio to the bound}."""
    cplan = pe.plan(net)
    gemm = plan["gemm"]
    n_pass = len(ut["frame"])
    sub = lambda units: {k: np.asarray(v)[units] for k, v in ut.items()}
    reads = {}                                 # buffer -> layers that read or write it
    for li, L in enumerate(gemm):
        for b in (L["a_buf"][0], L["a_buf"][1], L["res_buf"], L["out"]["buf"]):
            if b >= 0 and not (li == 0 and gen_first and b == plan["first"]["out"]["buf"]):
                reads.setdefault(b, set()).add(li)
    gathered = {}                              # buffer -> (units, logical [n, H, W, C] fp32) of the units some layer needs
    for b in sorted(reads):                    # one grid in host memory at a time
        units = np.array(sorted(set().union(*[set(sel[li]) for li in reads[b]])), np.int64)
        flat = read(b)
        gathered[b] = (units, grid_gather(plan["bufs"][b], flat, units).astype(np.float32))
        del flat

    def logical(b, units):
        have, data = gathered[b]
        return data[np.searchsorted(have, units)]

    ratios = {}
    for li, L in enumerate(gemm):
        units = np.asarray(sorted(sel[li]), np.int64)
        ctx = lambda u, wo: str(units[u]) if wo is None else where(L, n_pass, n_sm, int(units[u]), wo)
        bufs, errs = {}, None
        for b in {L["a_buf"][0], L["a_buf"][1], L["res_buf"]} - {-1}:
            if li == 0 and gen_first and b == plan["first"]["out"]["buf"]:
                v, S = pe.first(net, sub(units), raw, cond)
                a = v.astype(np.float16).astype(np.float32)
                bufs[b] = grid_scatter(cplan["bufs"][b], a)
                errs = {b: grid_scatter(cplan["bufs"][b], (ulp16(a) + C_ACC * S).astype(np.float32))}
            else:
                bufs[b] = grid_scatter(cplan["bufs"][b], logical(b, units))
        val, S, E = pe.layer(net, li, bufs, sub(units), raw, cond, errs)
        if L["out"]["buf"] < 0:
            got = np.asarray(den)[units][:, None, None, :]
            ref, bound = val[..., :got.shape[-1]], (C_ACC * S + E)[..., :got.shape[-1]]
        else:
            got = logical(L["out"]["buf"], units)
            C = got.shape[-1]
            ref, bound = val[..., :C], ulp16(val[..., :C]) + C_ACC * S[..., :C] + E[..., :C]
        ratios[L["name"]] = compare(L["name"], got, ref, bound, ctx)
    return ratios
