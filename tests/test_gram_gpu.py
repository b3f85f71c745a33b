"""The cross-statistic kernels of activation matching against fp64, elementwise, on every tap geometry their gates
admit: the TMA-fed fused Gram (csrc/gram_tma.cu, plb_gram_tma, called through ``ops.TmaGramPlan`` so that geometries
outside the Python gate are covered too), the packed route (plb_pack_split_pair + plb_gemm_grouped, alone and as one
grouped persistent launch), the gate between them, long contractions and CUDA-graph replay.

References are computed in fp64 on the GPU.  X and Y are the [C, K] row views of the two operands
(``ops.as_rows_view``); |X| is the elementwise absolute value, qa = sum x^2, sa = sum x and aa = sum |x| per row.
  * Gram, elementwise:  |G - X Y^T| <= TOL (|X| |Y|^T).
  * Row moments:  |q - sum x^2| <= TOL_Q sum x^2  and  |s - sum x| <= TOL_Q sum |x|, for both operands.
  * cdist, on the squared distance:  |D^2 - D64^2| <= TOL (qa_i + qb_j + 2 (|X| |Y|^T)_ij), with D finite and <= 0
    everywhere; on a tap with Y = X the diagonal sits inside the same bound around 0.
  * Correlation, with its first-order condition bound.  With the centred sums ca = qa - sa^2 / K, cb likewise,
        |C - C64| <= TOL B_ij,  B_ij = ((|X||Y|^T)_ij + |sa_i sb_j| / K) / sqrt(ca_i cb_j)
                                       + |C64_ij| (qa_i / ca_i + qb_j / cb_j) / 2.
    B grows with mean^2 / variance, so a large-mean unit is judged by the conditioning of the moment formula (a
    property of the formula, not a defect of the kernel) while a kernel error still cannot hide.  A dead unit (an
    all-zero row, ca = 0) is left out of the bound and must give exactly 0.
Every entry whose bound is 0 must be exact, and a NaN or infinite output fails every bar.

Measured over every case of this file on a B200 (1000 W power limit), the largest ratios are: Gram 1.35e-6, row
moments 4.2e-7, cdist 7.0e-7, correlation 6.6e-7 (printed at the end of a run with pytest -s).  The largest Gram
ratios are all on sums of one sign (the diagonal of a Y = X tap, large-mean data) and negative: the tensor core's fp32
accumulator truncates within each 64-k chain (ops.MAX_CHAIN_KB), -1.1e-6 on average over the diagonal of the C = 1000
Y = X case, half that with one-box chains; sign-mixed data stays at 2e-7.  TOL = 2.5e-6 leaves a margin of 1.85x over
the Gram and 3.5x over the statistics, TOL_Q = 1e-6 2.4x over the moments; a kernel that drops one of the three tf32
products is off by ~1e-4.

A work item accumulates in fp32 before its sums reach fp64 (the Gram once per chain in the promotion registers, the
moments per converter lane), so ``TmaGramPlan`` caps the contraction of one item at ops.TMA_MAX_K_PER_ITEM whatever
split count it is given.  The long-contraction tests ask for the automatic split choice and for one split on K up to
2^25 and hold both to TOL and TOL_Q; the growth is printed (pytest -s) and recorded in RESULTS.md.

Guards: every operand is a contiguous view into a larger buffer whose GUARD floats just before and just after it
hold NaN, so a read outside the tensor map shows up as NaN; the partial tiles are filled with NaN before a launch,
so a tile or split the kernel never writes shows up after the finalize; the moment buffers start at zero and the
kernel must add into them.
"""
import math
import random

import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = 2.5e-6
TOL_Q = 1e-6
PLB_ESIZE, PLB_EALIGN = -2, -3
GUARD = 64  # NaN floats on either side of an operand: 256 bytes, so an aligned operand stays 16-byte aligned
NAN = float("nan")
INNER, INNER_Q, CDIST, CORR = "inner", "inner+q", "cdist", "corr"
MAXIMA = {"gram": 0.0, "moments": 0.0, "cdist": 0.0, "corr": 0.0}


def _ops():
    from pleas_merging_b200 import ops

    return ops


def _launches(name):
    from pleas_merging_b200 import _native

    return _native.LAUNCH_COUNTS[name]


@pytest.fixture(scope="module", autouse=True)
def _report_maxima():
    yield
    print("\nlargest ratios over tests/test_gram_gpu.py: " + ", ".join(f"{k} {v:.3g}" for k, v in MAXIMA.items()))


# ------------------------------------------------------------------------------------------------ inputs


def _fill(x, kind, gen):
    """Fills the [outer, C, inner] tensor ``x`` in place with one input family."""
    C = x.shape[1]
    if kind == "lowbits":  # the 13 mantissa bits below tf32 all set, |x| in [0.25, 4), random signs
        bits = torch.randint(0, 1 << 23, x.shape, generator=gen, device=x.device, dtype=torch.int32)
        expo = torch.randint(125, 129, x.shape, generator=gen, device=x.device, dtype=torch.int32)
        x.copy_((bits | 0x1FFF | (expo << 23)).view(torch.float32))
        x.mul_(torch.randint(0, 2, x.shape, generator=gen, device=x.device).float().mul_(2).sub_(1))
        return
    x.normal_(generator=gen)
    if kind == "relu":
        x.relu_()
    elif kind == "mean":  # large mean against the spread: cdist and correlation cancel
        x.mul_(0.05).add_(4.0)
    elif kind == "scaled":  # rows scaled by 2^-20, 1, 2^20 in turn: only an elementwise bar sees the small ones
        e = torch.tensor([-20.0, 0.0, 20.0], device=x.device).repeat(C // 3 + 1)[:C]
        x.mul_(torch.exp2(e).view(1, C, *[1] * (x.dim() - 2)))
    elif kind == "dead":  # post-ReLU with every 7th unit all zero
        x.relu_()
        x[:, ::7].zero_()
    else:
        assert kind == "normal", kind


def _operand(shape, kind, seed, offset=0):
    """A contiguous [outer, C, inner] operand ``offset`` floats past a 16-byte boundary, inside a buffer whose GUARD
    floats just before and just after it hold NaN."""
    n = math.prod(shape)
    buf = torch.full((n + 2 * GUARD + offset,), NAN, device="cuda")
    x = buf[GUARD + offset:GUARD + offset + n].view(shape)
    _fill(x, kind, torch.Generator(device="cuda").manual_seed(seed))
    return x


def _pair(shape, kind, seed, offset=0):
    """(x, y): two independent draws, or the same tensor twice for kind "same-<family>"."""
    if kind.startswith("same-"):
        x = _operand(shape, kind[5:], seed, offset)
        return x, x
    return _operand(shape, kind, seed, offset), _operand(shape, kind, seed + 1, offset)


# ------------------------------------------------------------------------------------------------ references


def _reference(x, y, chunk=1 << 26):
    """fp64 G = X Y^T, A = |X| |Y|^T and the rows' moments [qa, sa, aa, qb, sb, ab] of an [outer, Ca, inner] and an
    [outer, Cb, inner] operand, accumulated over chunks of images."""
    outer, Ca, inner = x.shape
    Cb = y.shape[1]
    f64 = dict(dtype=torch.float64, device=x.device)
    G, A = torch.zeros(Ca, Cb, **f64), torch.zeros(Ca, Cb, **f64)
    mom = [torch.zeros(C, **f64) for C in (Ca, Ca, Ca, Cb, Cb, Cb)]
    step = max(1, chunk // (max(Ca, Cb) * inner))
    for o in range(0, outer, step):
        xa = x[o:o + step].double().transpose(0, 1).reshape(Ca, -1)
        yb = xa if y is x else y[o:o + step].double().transpose(0, 1).reshape(Cb, -1)
        G += xa @ yb.T
        A += xa.abs() @ yb.abs().T
        for k, r in enumerate((xa, yb)):
            mom[3 * k] += (r * r).sum(1)
            mom[3 * k + 1] += r.sum(1)
            mom[3 * k + 2] += r.abs().sum(1)
    return G, A, mom


def _ratio(err, bound):
    """max of err / bound; an entry whose bound is 0 must be exact, and a NaN or infinite error counts as inf."""
    err = torch.where(torch.isfinite(err), err, torch.full_like(err, math.inf))
    r = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, math.inf, 0.0))
    return r.max().item()


def _gram_ratio(G, G64, A):
    return _ratio((G.double() - G64).abs(), A)


def _moment_ratio(q, s, mom, which):
    """Ratio of the kernel's sums of squares q (and sums s, if given) of operand ``which`` (0 = x, 1 = y)."""
    q64, s64, a64 = mom[3 * which], mom[3 * which + 1], mom[3 * which + 2]
    r = _ratio((q - q64).abs(), q64)
    if s is not None:
        r = max(r, _ratio((s - s64).abs(), a64))
    return r


def _cdist_ratio(D, G64, A, mom):
    assert torch.isfinite(D).all() and (D <= 0).all()
    qa, qb = mom[0][:, None], mom[3][None]
    d2 = (qa + qb - 2 * G64).clamp_min(0)
    return _ratio((D.double() ** 2 - d2).abs(), qa + qb + 2 * A)


def _corr_ratio(Cc, G64, A, mom, K):
    qa, sa, qb, sb = mom[0], mom[1], mom[3], mom[4]
    ca, cb = qa - sa * sa / K, qb - sb * sb / K
    live = (qa > 0)[:, None] & (qb > 0)[None]
    assert torch.isfinite(Cc).all() and (Cc[~live] == 0).all(), "a dead unit must correlate with nothing, exactly"
    den = torch.sqrt(ca[:, None] * cb[None])
    C64 = (G64 - sa[:, None] * sb[None] / K) / den
    B = (A + (sa[:, None] * sb[None]).abs() / K) / den + C64.abs() * ((qa / ca)[:, None] + (qb / cb)[None]) / 2
    return _ratio(torch.where(live, (Cc.double() - C64).abs(), 0.0), torch.where(live, B, 1.0))


def _note(key, r):
    MAXIMA[key] = max(MAXIMA[key], r)
    return r


def _check_outputs(mode, G, out, G64, A, mom, K, q=None):
    """The bars of one tap: G (always), the statistic ``out`` of ``mode``, and the moments ``q`` = [qa, qb, sa, sb]
    the kernel accumulated (None: not requested)."""
    r = _note("gram", _gram_ratio(G, G64, A))
    assert r <= TOL, f"Gram: max |G - G64| / (|X||Y|^T) = {r:.3g} > {TOL:g}"
    if q is not None:
        sums = mode == CORR
        r = _note("moments", max(_moment_ratio(q[0], q[2] if sums else None, mom, 0),
                                 _moment_ratio(q[1], q[3] if sums else None, mom, 1)))
        assert r <= TOL_Q, f"row moments: ratio {r:.3g} > {TOL_Q:g}"
    if mode == CDIST:
        r = _note("cdist", _cdist_ratio(out, G64, A, mom))
        assert r <= TOL, f"cdist: ratio {r:.3g} > {TOL:g}"
    elif mode == CORR:
        r = _note("corr", _corr_ratio(out, G64, A, mom, K))
        assert r <= TOL, f"correlation: ratio {r:.3g} > {TOL:g}"


def _mode_code(mode):
    ops = _ops()
    return {INNER: ops.MODE_INNER, INNER_Q: ops.MODE_INNER, CDIST: ops.MODE_NEG_CDIST, CORR: ops.MODE_CORR}[mode]


# ------------------------------------------------------------------------------------------------ the TMA route


def _total_boxes(outer, inner):
    return outer * ((inner + 31) // 32)


def _run_tma(x, y, splits, mode):
    """One plb_gram_tma launch through TmaGramPlan on NaN-filled partial tiles and zeroed moments, then the finalize
    of ``mode`` and of the plain Gram.  Returns (G, statistic, moments [qa, qb, sa, sb] or None, plan)."""
    ops = _ops()
    outer, C, inner = x.shape
    if splits == "all":
        splits = _total_boxes(outer, inner)
    plan = ops.TmaGramPlan(C, outer, inner, x.device, splits=splits)
    plan.partial.fill_(NAN)
    q = torch.zeros(4, C, dtype=torch.float64, device=x.device) if mode != INNER else None
    qa, qb = (q[0], q[1]) if q is not None else (None, None)
    sa, sb = (q[2], q[3]) if mode == CORR else (None, None)
    before = _launches("plb_gram_tma")
    plan.run(x, y, 1, qa, qb, sa, sb)
    assert _launches("plb_gram_tma") == before + 1
    G = torch.empty(C, C, device=x.device)
    plan.finalize(G, ops.MODE_INNER)
    out = G
    if mode in (CDIST, CORR):
        out = torch.empty(C, C, device=x.device)
        plan.finalize(out, _mode_code(mode), qa, qb, sa=sa, sb=sb, K=outer * inner)
    return G, out, q, plan


TMA_CASES = [
    # (C, outer, inner, splits, input, statistic); splits None = choose_tma_splits, "all" = one box per work item
    (8, 256, 4, None, "normal", INNER_Q),
    (9, 31, 8, 1, "relu", CDIST),             # outer * inner = 248 < 256
    (63, 3, 12, "all", "mean", CORR),
    (64, 16, 16, 2, "lowbits", INNER),        # outer * inner = 256
    (65, 31, 20, 5, "scaled", CDIST),
    (127, 1, 28, 1, "dead", CORR),            # one box in all
    (128, 2, 32, "all", "normal", INNER_Q),
    (129, 3, 36, None, "relu", CORR),         # pair tile: the second CTA holds 1 valid row; 4 valid k in box 2
    (200, 256, 48, None, "mean", CDIST),      # second CTA: 72 rows
    (255, 31, 60, 2, "lowbits", INNER_Q),     # second CTA: 127 rows
    (256, 1, 196, 1, "scaled", CORR),
    (257, 2, 784, 5, "dead", CDIST),          # a second 256-row tile holding one row
    (384, 1, 3136, None, "normal", INNER),    # the second CTA of tile 2 holds no row at all
    (513, 1, 12544, 3, "relu", CORR),
    (1000, 3, 196, None, "same-normal", CDIST),
    (2048, 2, 196, 2, "relu", INNER_Q),       # 128 work items on 74 clusters
    (4096, 2, 36, 1, "normal", INNER),        # 256 work items on 74 clusters
    (64, 1, 12544, "all", "relu", INNER_Q),   # 392 one-box work items on 148 CTAs
    (8, 1, 3136, None, "same-relu", CORR),
    (200, 31, 4, 1, "normal", INNER_Q),
    (129, 256, 8, None, "dead", CORR),
    (255, 2, 12, "all", "same-mean", CORR),
    (64, 256, 28, None, "normal", CDIST),
    (1000, 31, 16, None, "lowbits", CORR),
    (128, 3, 60, 5, "scaled", INNER_Q),
    (9, 2, 196, 7, "mean", CORR),
    (384, 256, 20, None, "relu", CDIST),
    (63, 31, 36, 7, "same-scaled", CDIST),
    (513, 2, 48, "all", "same-dead", CORR),
]


def _tma_case(case, seed):
    C, outer, inner, splits, kind, mode = case
    x, y = _pair((outer, C, inner), kind, seed)
    G, out, q, plan = _run_tma(x, y, splits, mode)
    G64, A, mom = _reference(x, y)
    # with Y = X the cdist bar holds the diagonal to the same bound around 0
    _check_outputs(mode, G, out, G64, A, mom, outer * inner, q)
    return x, y, plan, q


@pytest.mark.parametrize("case", TMA_CASES, ids=[str(c) for c in TMA_CASES])
def test_tma_route_matches_fp64(case):
    _tma_case(case, seed=1000 + TMA_CASES.index(case))


@pytest.mark.parametrize("chain", [1, 2, 4])
@pytest.mark.parametrize("case", [(200, 31, 60, None, "normal", CDIST), (64, 3, 784, 1, "relu", CORR),
                                  (513, 2, 196, 2, "mean", CORR)], ids=str)
def test_tma_route_chain_lengths(case, chain, monkeypatch):
    """Chains of 1, 2 and 4 k-blocks (one or two boxes) between promotions into the fp32 registers."""
    monkeypatch.setattr(_ops(), "MAX_CHAIN_KB", chain)
    _tma_case(case, seed=2000 + chain)


def test_tma_moments_accumulate():
    """plb_gram_tma adds its row moments into the caller's buffers (a calibration batch sums several taps and
    batches into them): a second launch doubles them."""
    x, y, plan, q = _tma_case((200, 3, 196, 3, "relu", CORR), seed=3000)
    first = q.clone()
    qa, qb, sa, sb = q
    plan.run(x, y, 1, qa, qb, sa, sb)
    torch.testing.assert_close(q, 2 * first, rtol=1e-12, atol=0)


# ------------------------------------------------------------------------------------------------ long contractions

LONG_CASES = [  # (C, outer, inner): K from about 2^16 to about 2^25 by growing the batch
    (64, 2, 50176), (64, 10, 50176), (64, 84, 50176), (64, 700, 50176),  # the last: 2.2e9 elements per operand
    (256, 21, 3136), (256, 167, 3136), (256, 1337, 3136), (256, 10700, 3136),
]


@pytest.mark.parametrize("C,outer,inner", LONG_CASES, ids=str)
def test_tma_long_contraction(C, outer, inner):
    """Accuracy against the length of the contraction: the automatic split choice and a request for one split both
    meet TOL and TOL_Q at every size, because no work item walks more than TMA_MAX_K_PER_ITEM of K."""
    ops = _ops()
    x, y = _pair((outer, C, inner), "relu", 4000 + C + outer)
    G64, A, mom = _reference(x, y)
    K, boxes = outer * inner, _total_boxes(outer, inner)
    rows = []
    for splits in (None, 1):
        G, _, q, plan = _run_tma(x, y, splits, CORR)
        rg = _gram_ratio(G, G64, A)
        rq = max(_moment_ratio(q[0], None, mom, 0), _moment_ratio(q[1], None, mom, 1))
        rs = max(_ratio((q[2] - mom[1]).abs(), mom[2]), _ratio((q[3] - mom[4]).abs(), mom[5]))
        rows.append((plan.splits, rg, rq, rs))
        assert -(-boxes // plan.splits) * 32 <= ops.TMA_MAX_K_PER_ITEM, plan.splits
        del G, plan
    print(f"\nlong K: C {C} K {K} (2^{math.log2(K):.1f}) boxes {boxes}: " + "; ".join(
        f"splits {s} ({boxes / s:.0f} boxes/item): gram {rg:.3g} sumsq {rq:.3g} sum {rs:.3g}" for s, rg, rq, rs in rows))
    for _, rg, rq, rs in rows:
        _note("gram", rg)
        _note("moments", max(rq, rs))
        assert rg <= TOL and max(rq, rs) <= TOL_Q, rows


# ------------------------------------------------------------------------------------------------ packed route + gate


def _cross(x, y, axis, mode):
    """ops.cross_statistic for ``mode``, the plain Gram, and the fp64 references on the [outer, C, inner] views."""
    ops = _ops()
    G = ops.cross_statistic(x, y, axis, ops.MODE_INNER)
    out = ops.cross_statistic(x, y, axis, _mode_code(mode)) if mode in (CDIST, CORR) else G
    shape = ops.as_rows_view(x, axis)
    xs = x.reshape(shape)
    G64, A, mom = _reference(xs, xs if y is x else y.reshape(shape))
    return G, out, G64, A, mom, shape[0] * shape[2]


PACKED_CASES = [
    # (shape, axis, input, pointer offset in floats)
    ((32, 512, 7, 7), 1, "relu", 0),        # the two most expensive packed classes of a ResNet-50 step
    ((32, 2048, 7, 7), 1, "relu", 0),
    ((4, 64, 3, 3), 1, "normal", 0),        # inner 9
    ((3, 100, 5, 5), 1, "mean", 0),         # inner 25
    ((5, 40, 2, 3), 1, "dead", 0),          # inner 6
    ((64, 300), 1, "relu", 0),              # flat [B, C]: inner 1
    ((96, 1000), 1, "same-scaled", 0),
    ((4, 1, 16, 16), 1, "normal", 0),       # C from 1 to 7
    ((2, 3, 8, 8), 1, "lowbits", 0),
    ((3, 7, 12, 12), 1, "same-mean", 0),
    ((2, 5, 20), 1, "dead", 0),
    ((2, 64, 16, 16), 1, "relu", 1),        # 4, 8 and 12 bytes past a 16-byte boundary
    ((3, 256, 14, 14), 1, "mean", 2),
    ((2, 8, 8, 8), 1, "normal", 3),
    ((4, 130, 6, 6), 1, "scaled", 1),
]


@pytest.mark.parametrize("shape,axis,kind,offset", PACKED_CASES, ids=str)
def test_packed_route_matches_fp64(shape, axis, kind, offset):
    """Taps the TMA gate refuses run pack + 3xTF32 GEMM (no plb_gram_tma launch) and meet the same bars."""
    ops = _ops()
    x, y = _pair(shape, kind, 5000 + len(shape) + shape[1], offset)
    assert not ops.tma_gram_eligible(x, y, axis)
    before = {n: _launches(n) for n in ("plb_gram_tma", "plb_pack_split_pair_sums", "plb_gemm_grouped")}
    for mode in (INNER, CDIST, CORR):
        G, out, G64, A, mom, K = _cross(x, y, axis, mode)
        _check_outputs(mode, G, out, G64, A, mom, K)
    assert _launches("plb_gram_tma") == before["plb_gram_tma"]
    assert _launches("plb_pack_split_pair_sums") == before["plb_pack_split_pair_sums"] + 5
    assert _launches("plb_gemm_grouped") == before["plb_gemm_grouped"] + 5


GATE_SHAPES = [(8, 16, 12), (64, 9, 8), (3, 130, 20), (20, 8, 36), (2, 40, 6), (256, 1, 8), (48, 64), (9, 4, 64)]


@pytest.mark.parametrize("offset", [0, 2])
@pytest.mark.parametrize("shape", GATE_SHAPES, ids=str)
def test_gate_and_routes_agree(shape, offset):
    """Over C, inner, outer, pointer offset and axis: wherever tma_gram_eligible holds, cross_statistic launches
    plb_gram_tma exactly once, elsewhere never, and both routes meet the bars."""
    ops = _ops()
    x, y = _pair(shape, "relu", 6000 + sum(shape) + offset, offset)
    for axis in range(len(shape)):
        mode = (INNER, CDIST, CORR)[(axis + offset) % 3]
        eligible = ops.tma_gram_eligible(x, y, axis)
        before = _launches("plb_gram_tma")
        G, out, G64, A, mom, K = _cross(x, y, axis, mode)
        calls = 1 if mode == INNER else 2
        assert _launches("plb_gram_tma") == before + (calls if eligible else 0), (axis, eligible)
        _check_outputs(mode, G, out, G64, A, mom, K)


def test_tma_entry_point_refuses_what_its_gate_refuses():
    """plb_gram_tma refuses inner % 4 != 0 with PLB_ESIZE and a misaligned operand or partial pointer with
    PLB_EALIGN, and launches nothing: the partial tiles stay NaN and the moments zero."""
    ops = _ops()
    lib = ops.N.lib()
    stream = torch.cuda.current_stream().cuda_stream
    partial = torch.full(((1 << 16) + 4,), NAN, device="cuda")
    q = torch.zeros(4, 64, dtype=torch.float64, device="cuda")
    qp = [t.data_ptr() for t in q]

    def call(x, y, outer, C, inner, part):
        rc = lib.plb_gram_tma(x.data_ptr(), y.data_ptr(), outer, C, inner, part, 1, ops.MAX_CHAIN_KB, *qp, stream)
        torch.cuda.synchronize()
        return rc

    x, y = _pair((4, 64, 6), "normal", 7000)
    assert call(x, y, 4, 64, 6, partial.data_ptr()) == PLB_ESIZE
    xa, ya = _pair((4, 64, 16), "normal", 7001)
    xm, ym = _pair((4, 64, 16), "normal", 7002, offset=1)
    assert call(xm, ya, 4, 64, 16, partial.data_ptr()) == PLB_EALIGN
    assert call(xa, ym, 4, 64, 16, partial.data_ptr()) == PLB_EALIGN
    assert call(xa, ya, 4, 64, 16, partial.data_ptr() + 8) == PLB_EALIGN
    assert torch.isnan(partial).all() and (q == 0).all()
    assert call(xa, ya, 4, 64, 16, partial.data_ptr()) == 0  # the same operands, aligned: accepted


# ------------------------------------------------------------------------------------------------ grouped launch


def _grouped_problems(bn, n, seed):
    """n (M, N, K) of one tile width ``bn``: M over one or two 128-row tiles, N in bn's class, K from one k-block to
    a few thousand; the first problem takes a single CTA."""
    rng = random.Random(seed)
    lo_n = {64: 1, 128: 65, 256: 129}[bn]
    probs = [(rng.randint(1, 128), rng.randint(lo_n, bn), rng.randint(1, 1000))]
    for _ in range(n - 1):
        probs.append((rng.randint(1, 256), rng.randint(lo_n, bn), rng.choice([16, 500, 2050, 6000, 12345])))
    return probs


def _grouped_setup(bn, n, seed):
    """Packed operands and a GemmPlan per problem (the deferred taps' split rule), on NaN-filled partial tiles."""
    ops = _ops()
    plans, data = [], []
    for i, (M, Nn, K) in enumerate(_grouped_problems(bn, n, seed)):
        xa = _operand((1, M, K), "relu" if i % 2 else "normal", seed + 2 * i)
        xb = _operand((1, Nn, K), "normal" if i % 3 else "mean", seed + 2 * i + 1)
        kb = (K + 15) // 16
        pa, pb = ops.Planes(M, kb, xa.device), ops.Planes(Nn, kb, xa.device)
        plan = ops.GemmPlan(pa, pb, M, Nn, kb, splits=max(1, min(kb // 32, 16)))
        assert plan.bn == bn
        plan.partial.fill_(NAN)
        plans.append(plan)
        data.append((xa, xb, pa, pb))
    if n > 1:
        assert plans[0].total_ctas == 1
    return plans, data


def _pack_all(data):
    ops = _ops()
    for xa, xb, pa, pb in data:
        ops.pack_split(xa, 1, pa)
        ops.pack_split(xb, 1, pb)


def _partials(plan):
    """The [splits, M, N] region of a plan's partial tiles, as raw bits."""
    t = plan.partial[:plan.splits * plan.ld_m * plan.ld_n].view(plan.splits, plan.ld_m, plan.ld_n)
    return t[:, :plan.M, :plan.N].view(torch.int32).clone()


@pytest.mark.parametrize("n", [2, 5, 17])
@pytest.mark.parametrize("bn", [64, 128, 256])
def test_grouped_launch_equals_single_launches(bn, n):
    """Problems of one tile width in one persistent launch (the route of the deferred small taps): every problem's
    partial tiles are bit-equal to a launch of that problem alone, and every finalized Gram meets the fp64 bar."""
    ops = _ops()
    plans, data = _grouped_setup(bn, n, 8000 + bn + n)
    _pack_all(data)
    alone = []
    for p in plans:
        p.run()
        alone.append(_partials(p))
        p.partial.fill_(NAN)
    before = _launches("plb_gemm_grouped")
    ops.GroupedGemm(plans).run()
    assert _launches("plb_gemm_grouped") == before + 1
    for p, ref, (xa, xb, _, _) in zip(plans, alone, data):
        assert torch.equal(_partials(p), ref), (p.M, p.N, p.splits)
        G = torch.empty(p.M, p.N, device="cuda")
        p.finalize(G)
        G64, A, _ = _reference(xa, xb)
        r = _note("gram", _gram_ratio(G, G64, A))
        assert r <= TOL, (p.M, p.N, p.splits, r)


# ------------------------------------------------------------------------------------------------ graph replay


def _captured(fn):
    fn()  # eager warm-up: kernel attributes and modules are set before the capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g


def test_graph_replay_tma_tap_is_bit_equal():
    """A TMA-route tap captured in a CUDA graph (as the calibration runner runs it) and replayed on new data in the
    same buffers gives the eager launch's Gram bit for bit."""
    ops = _ops()
    outer, C, inner = 6, 320, 196
    x, y = _pair((outer, C, inner), "relu", 9000)
    plan = ops.TmaGramPlan(C, outer, inner, x.device)
    q = torch.zeros(4, C, dtype=torch.float64, device="cuda")
    G = torch.empty(C, C, device="cuda")

    def tap():
        q.zero_()
        plan.run(x, y, 1, q[0], q[1], q[2], q[3])
        plan.finalize(G, ops.MODE_INNER)

    g = _captured(tap)
    _fill(x, "mean", torch.Generator(device="cuda").manual_seed(9001))
    _fill(y, "normal", torch.Generator(device="cuda").manual_seed(9002))
    before = _launches("plb_gram_tma")
    g.replay()
    assert _launches("plb_gram_tma") == before  # a replay does not go through the host
    replayed, q_replayed = G.clone(), q.clone()
    tap()
    assert torch.equal(replayed, G)
    G64, A, mom = _reference(x, y)
    assert _gram_ratio(replayed, G64, A) <= TOL
    assert max(_moment_ratio(q_replayed[0], q_replayed[2], mom, 0), _moment_ratio(q_replayed[1], q_replayed[3], mom, 1)) <= TOL_Q


def test_graph_replay_grouped_launch_is_bit_equal():
    """Packing and one grouped persistent launch captured in a CUDA graph and replayed on new data give the eager
    launch's partial tiles bit for bit."""
    ops = _ops()
    plans, data = _grouped_setup(128, 5, 9100)
    grouped = ops.GroupedGemm(plans)

    def step():
        _pack_all(data)
        grouped.run()

    g = _captured(step)
    for i, (xa, xb, _, _) in enumerate(data):
        _fill(xa, "dead", torch.Generator(device="cuda").manual_seed(9200 + i))
        _fill(xb, "scaled", torch.Generator(device="cuda").manual_seed(9300 + i))
    g.replay()
    replayed = [_partials(p) for p in plans]
    for p in plans:
        p.partial.fill_(NAN)
    step()
    for p, r, (xa, xb, _, _) in zip(plans, replayed, data):
        assert torch.equal(_partials(p), r)
        G = torch.empty(p.M, p.N, device="cuda")
        p.finalize(G)
        G64, A, _ = _reference(xa, xb)
        assert _gram_ratio(G, G64, A) <= TOL
