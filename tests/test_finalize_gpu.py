"""The cost epilogue of activation matching (csrc/finalize.cu) against fp64, elementwise, and the accuracy of
derived BatchNorm taps against contracted ones.

1. plb_cross_finalize_grouped, called directly on tap and group tables built with ``ops.N`` and ``ops.TableArena``,
   on synthetic K-split partial tiles: X and Y are random [n, K] matrices of fp32 values, the partial tile of split s
   is X_s Y_s^T over that split's columns rounded to fp32, and qa = sum x^2, sa = sum x are formed in fp64.  The
   reference sums the same fp32 partials in fp64 (G) and applies each statistic in fp64, so it is exact to 2^-50.
   Bars, per cost entry, with u = 2^-24 and |.| elementwise:
     * inner:  u |G| per tap; a derived tap  u |w| + 2^-48 (sum of the |terms| of its formula);
     * cdist:  the fp32 formula (float)qa + (float)qb - 2 (float)G bounds d^2 by E = 4u (qa + qb + 2|G|) (a derived
       tap: E = u |d^2| + 2^-48 (sum of |terms|)), and d = sqrt(d^2) follows within min(sqrt(E), E / d) + u d;
     * corr:   u |C| + 2^-48 (its first-order condition number), and exactly 0 for a unit without variance;
   plus u (T + 1) (sum over the T values added of |value|) for the fp32 adds across taps and into the cost entry.
   Each bar is a worst-case rounding bound, which many entries approach; it is applied with a factor SLACK = 1.5.
   The cost entries outside [n][n] but inside ldc, and the fp32 words around every cost matrix, hold a sentinel that
   must be bit-unchanged; the partial padding, one split past ``splits`` and the words around every moment and
   affine vector hold NaN, so a read outside the data shows up in the result.
   The per-tap kernels reached through ``GemmPlan.finalize`` (plb_cross_finalize, its stream / reduce switch at
   48 / 49 splits, fp64 output and the symmetric tile mask; plb_cross_finalize_corr) are held to the same bars.

2. Derived BatchNorm taps against contracted ones.  The real Gram kernel (``ops.TmaGramPlan``) contracts fp32 X and Y
   with controlled per-unit mean / spread mu / sigma, and the grouped epilogue derives the statistic of the
   BatchNorm outputs x' = s x + t (n_affine = 1), with (s, t) from the batch statistics and beta / gamma chosen.  The
   contracted route runs the same kernels on x' materialised in fp32.  Both are held to the contracted route's bars
   of tests/test_gram_gpu.py, computed from x' in fp64: the derived error grows like kappa_a kappa_b / (kappa'_a
   kappa'_b) (activation_matching.BN_AFFINE_MAX_GROWTH), so only the derivations that bound admits must meet them.
   ``pytest -s`` prints the table of ratios; RESULTS.md records it.
"""
import math

import pytest
import torch

from test_gram_gpu import TOL, _cdist_ratio, _corr_ratio, _ratio, _reference

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
E64 = 2.0 ** -48  # allowance for fp64 evaluation order (kernel and reference differ in the order of their terms)
GUARD = 64
NAN = float("nan")
SENTINEL = -1.2345e30
SLACK = 1.5
AFFINE_GUARD = 1024  # NaN doubles behind the affine vectors: room for a kernel that strides them by ldc instead of n
INNER, CDIST, CORR = "inner", "cdist", "corr"
MAXIMA = {"grouped": 0.0, "per-tap": 0.0}
COND_TABLE = []


def _ops():
    from pleas_merging_b200 import ops

    return ops


def _am():
    import importlib

    return importlib.import_module("pleas_merging_b200.methods.activation_matching")


def _launches(name):
    from pleas_merging_b200 import _native

    return _native.LAUNCH_COUNTS[name]


def _mode_code(mode):
    ops = _ops()
    return {INNER: ops.MODE_INNER, CDIST: ops.MODE_NEG_CDIST, CORR: ops.MODE_CORR}[mode]


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print("\nlargest ratios over tests/test_finalize_gpu.py: " + ", ".join(f"{k} {v:.3g}" for k, v in MAXIMA.items()))
    if COND_TABLE:
        print("derived vs contracted BatchNorm taps (ratio to the contracted route's bar):")
        print("  mu/sigma  beta/gamma  gamma<0  mode   growth      derived   contracted  admitted")
        for mu, bg, neg, mode, growth, rd, rc, ok in sorted(COND_TABLE, key=lambda r: (r[3], r[2], r[0], r[1])):
            print(f"  {mu:8g}  {bg:10g}  {str(neg):7s}  {mode:5s}  {growth:9.4g}  {rd:10.3g}  {rc:10.3g}  {ok}")


def _note(key, r):
    MAXIMA[key] = max(MAXIMA[key], r)
    return r


# ------------------------------------------------------------------------------------------------ guarded buffers


def _guarded(n, dtype, fill):
    """A length-n view with GUARD elements of ``fill`` on either side (256 bytes or more: alignment is kept)."""
    buf = torch.full((n + 2 * GUARD,), fill, dtype=dtype, device="cuda")
    return buf[GUARD:GUARD + n], buf


def _guarded64(values, tail=0):
    v, _ = _guarded(values.numel() + tail, torch.float64, NAN)
    v = v[:values.numel()]
    v.copy_(values.reshape(-1))
    return v


# ------------------------------------------------------------------------------------------------ synthetic taps


def _layout(n, layout):
    """(ld_m, ld_n) of the partial tiles that production plans allocate for an n-unit tap."""
    ops = _ops()
    if layout == "gemm":
        bn = ops.choose_bn(n)
        return (n + 127) // 128 * 128, (n + bn - 1) // bn * bn
    if layout == "direct":
        assert n <= 128
        return 128, 64 if n <= 64 else 128
    if layout in ("tma1", "tma2"):
        cg, _, _, ld_m, ld_n = ops.tma_geometry(n)
        assert cg == int(layout[-1]), (n, cg)
        return ld_m, ld_n
    assert layout == "wide"  # padded past any plan: rows and 64 columns of NaN beyond the data
    return n + 37, (n + 63) // 64 * 64 + 64


def _rows(n, K, kind, gen):
    """[n, K] fp64 matrix of fp32 values of one input family."""
    x = torch.randn(n, K, generator=gen, device="cuda", dtype=torch.float64)
    if kind == "mean":  # large mean against the spread: cdist and correlation cancel
        x = 4.0 + 0.05 * x
    elif kind == "dead":  # every 7th unit all zero
        x = x.relu()
        x[::7] = 0.0
    else:
        assert kind == "normal", kind
    return x.float().double()


class _Tap:
    """One tap of a group: partial tiles in a NaN-guarded [splits + 1][ld_m][ld_n] buffer, guarded fp64 moments and
    affine vectors, and the fp64 quantities the reference needs."""

    def __init__(self, n, splits, layout, n_affine, kind, seed):
        gen = torch.Generator(device="cuda").manual_seed(seed)
        kc = max(1, 12 // splits)
        K = splits * kc
        X, Y = _rows(n, K, kind, gen), _rows(n, K, "dead" if kind == "dead" else "normal", gen)
        if kind == "dead":
            Y[3::5] = 0.0
        self.n, self.K, self.splits, self.n_affine = n, K, splits, n_affine
        self.ld_m, self.ld_n = _layout(n, layout) if isinstance(layout, str) else layout
        self.partial, _ = _guarded((splits + 1) * self.ld_m * self.ld_n, torch.float32, NAN)
        P = self.partial.view(splits + 1, self.ld_m, self.ld_n)
        G, Pabs = torch.zeros(n, n, dtype=torch.float64, device="cuda"), torch.zeros(n, n, dtype=torch.float64,
                                                                                      device="cuda")
        for s in range(splits):
            p = (X[:, s * kc:(s + 1) * kc] @ Y[:, s * kc:(s + 1) * kc].T).float()
            P[s, :n, :n] = p
            G += p.double()
            Pabs += p.double().abs()
        self.G, self.Pabs = G, Pabs
        self.qa64, self.qb64 = (X * X).sum(1), (Y * Y).sum(1)
        self.sa64, self.sb64 = X.sum(1), Y.sum(1)
        self.qa, self.qb, self.sa, self.sb = (_guarded64(v) for v in (self.qa64, self.qb64, self.sa64, self.sb64))
        self.aff64 = []
        for _ in range(n_affine):  # s of both signs and exactly 0 on every 5th unit; |t| ~ 300 |s| on every 3rd
            vecs = []
            for _side in range(2):
                s = torch.randn(n, generator=gen, device="cuda", dtype=torch.float64)
                s[::5] = 0.0
                t = torch.randn(n, generator=gen, device="cuda", dtype=torch.float64)
                t[::3] *= 300.0
                vecs += [s, t]
            self.aff64.append(vecs)
        self.affine = _guarded64(torch.cat([v for vecs in self.aff64 for v in vecs]), AFFINE_GUARD) \
            if n_affine else None

    def entry(self):
        ops = _ops()
        return ops.N.FinalizeTap(self.partial.data_ptr(), self.qa.data_ptr(), self.qb.data_ptr(), self.sa.data_ptr(),
                                 self.sb.data_ptr(), self.ld_m, self.ld_n, self.K, self.splits, self.n_affine,
                                 ops.N.ptr(self.affine))

    def values(self, mode):
        """[(value, bar)] in fp64 for the tap's own statistic and each derived one, in the kernel's order."""
        G, Pabs, K = self.G, self.Pabs, self.K
        qa, qb, sa, sb = self.qa64[:, None], self.qb64[None], self.sa64[:, None], self.sb64[None]
        out = []
        if mode == INNER:
            out.append((G, U * G.abs() + E64 * Pabs))
        elif mode == CDIST:
            d2 = qa + qb - 2 * G
            out.append(_dist(d2, 4 * U * (qa + qb + 2 * G.abs()) + E64 * 2 * Pabs))
        else:
            va, vb = qa - sa * sa / K, qb - sb * sb / K
            live = (va > 1e-12 * qa) & (vb > 1e-12 * qb)
            den = torch.sqrt((va * vb).clamp_min(1e-300))
            C = torch.where(live, (G - sa * sb / K) / den, 0.0)
            cond = (G.abs() + Pabs + (sa * sb).abs() / K) / den + C.abs() * (qa / va.clamp_min(1e-300) +
                                                                              qb / vb.clamp_min(1e-300))
            corr = (C, torch.where(live, U * C.abs() + E64 * cond, 0.0))
            out.append(corr)
        for s_a, t_a, s_b, t_b in self.aff64:
            s_a, t_a, s_b, t_b = s_a[:, None], t_a[:, None], s_b[None], t_b[None]
            if mode == INNER:
                terms = [s_a * s_b * G, s_a * t_b * sa, t_a * s_b * sb, K * t_a * t_b]
                w = sum(terms)
                out.append((w, U * w.abs() + E64 * (sum(t.abs() for t in terms) + (s_a * s_b).abs() * Pabs)))
            elif mode == CDIST:
                dt = t_a - t_b
                terms = [s_a * s_a * qa, s_b * s_b * qb, -2 * s_a * s_b * G, K * dt * dt,
                         2 * dt * (s_a * sa - s_b * sb)]
                d2 = sum(terms)
                out.append(_dist(d2, U * d2.abs() + E64 * (sum(t.abs() for t in terms) +
                                                           2 * (s_a * s_b).abs() * Pabs)))
            else:
                sg = torch.sign(s_a * s_b)
                out.append((sg * corr[0], sg.abs() * corr[1]))
        return out


def _dist(d2, E):
    """(-d, bar on d) from the squared distance d2 and the bound E on its error."""
    d = d2.clamp_min(0).sqrt()
    return -d, torch.minimum(E.sqrt(), E / d.clamp_min(1e-300)) + U * d


class _Group:
    """One permutation group's fp32 cost matrix [n][ldc] inside a sentinel-guarded buffer, and its taps."""

    def __init__(self, n, ldc_extra, taps, accumulate, seed):
        self.n, self.ldc, self.taps = n, n + ldc_extra, taps
        self.cost_flat, self.buf = _guarded(n * self.ldc, torch.float32, SENTINEL)
        self.cost = self.cost_flat.view(n, self.ldc)
        gen = torch.Generator(device="cuda").manual_seed(seed)
        # accumulate: random old entries; overwrite: NaN, so an entry the kernel never writes fails its bar
        self.cost[:, :n] = torch.randn(n, n, generator=gen, device="cuda") if accumulate else NAN
        self.old = self.cost[:, :n].double().clone() if accumulate else None
        self.before = self.buf.clone()

    def check(self, mode):
        """max ratio of |cost - reference| to the bar, after asserting every word outside [n][n] is bit-unchanged."""
        n = self.n
        mask = torch.ones_like(self.buf, dtype=torch.bool)
        mask[GUARD:GUARD + n * self.ldc].view(n, self.ldc)[:, :n] = False
        assert torch.equal(self.buf[mask].view(torch.int32), self.before[mask].view(torch.int32)), \
            "the kernel wrote outside [n][n] of a cost matrix"
        vals = [vb for tap in self.taps for vb in tap.values(mode)]
        ref = sum(v for v, _ in vals)
        mag = sum(v.abs() for v, _ in vals)
        bar = sum(b for _, b in vals) + U * len(vals) * mag
        if self.old is not None:
            ref = ref + self.old
            bar = bar + U * (mag + self.old.abs())
        got = self.cost[:, :n].double()
        return _ratio((got - ref).abs(), SLACK * bar)


def _run_grouped(groups, mode, accumulate):
    """One plb_cross_finalize_grouped launch over ``groups`` (tables through ops.TableArena)."""
    ops = _ops()
    taps_raw, groups_raw, blocks, t0 = bytearray(), bytearray(), 0, 0
    for g in groups:
        for tap in g.taps:
            taps_raw += bytes(tap.entry())
        groups_raw += bytes(ops.N.FinalizeGroup(g.cost.data_ptr(), g.ldc, g.n, t0, t0 + len(g.taps), blocks))
        t0 += len(g.taps)
        blocks += ops.finalize_grouped_blocks(g.n)
    arena = ops.TableArena("cuda")
    taps_t, groups_t = arena.put(bytes(taps_raw)), arena.put(bytes(groups_raw))
    before = _launches("plb_cross_finalize_grouped")
    ops.N.call("plb_cross_finalize_grouped", taps_t.device, taps_t.data_ptr(), groups_t.data_ptr(), len(groups),
               blocks, _mode_code(mode), int(accumulate))
    torch.cuda.synchronize()
    assert _launches("plb_cross_finalize_grouped") == before + 1


def _grouped_case(group_specs, mode, accumulate, seed):
    """group_specs: [(n, ldc_extra, [(splits, layout, n_affine, kind), ...]), ...].  Runs and checks every group."""
    groups = []
    for gi, (n, extra, tap_specs) in enumerate(group_specs):
        taps = [_Tap(n, sp, lay, na, kind, seed + 100 * gi + ti) for ti, (sp, lay, na, kind) in enumerate(tap_specs)]
        groups.append(_Group(n, extra, taps, accumulate, seed + 100 * gi + 99))
    _run_grouped(groups, mode, accumulate)
    worst = 0.0
    for g in groups:
        r = _note("grouped", g.check(mode))
        assert r <= 1.0, f"group n={g.n} ldc={g.ldc} {mode} accumulate={accumulate}: ratio {r:.3g}"
        worst = max(worst, r)
    return worst


# ------------------------------------------------------------------------------------------------ 1. grouped epilogue

GROUP_SIZES = [1, 3, 4, 5, 63, 64, 65, 255, 256, 257, 1000, 2048, 4096]


@pytest.mark.parametrize("n", GROUP_SIZES)
def test_grouped_tile_geometry(n):
    """One group of n units on either side of the switch from 64 x 64 to 256 x 16 tiles, n not a multiple of 4,
    ldc > n: two taps (odd and even splits, different layouts, one with a derived tap), every mode, overwrite and
    accumulate."""
    big = n > 1000
    taps = [(3, "gemm", 1, "normal"), (2 if big else 48, "wide", 0, "mean")]
    for k, mode in enumerate((INNER, CDIST, CORR)):
        for accumulate in (0, 1):
            _grouped_case([(n, 5 + 64 * accumulate, taps)], mode, accumulate, seed=10 * n + 2 * k + accumulate)


MIXED = [(5, 3, [(1, "gemm", 0, "normal")]), (300, 0, [(2, "tma2", 1, "mean"), (1, "gemm", 0, "normal")]),
         (1, 1, [(7, "wide", 2, "normal")]), (64, 0, [(3, "direct", 0, "dead")]),
         (257, 9, [(49, "gemm", 1, "normal")]), (63, 2, [(1, "tma1", 1, "mean"), (200, "wide", 0, "normal")]),
         (1000, 4, [(3, "tma2", 0, "normal")]), (4, 0, [(1, "direct", 1, "normal")]),
         (256, 0, [(5, "gemm", 0, "dead")])]


@pytest.mark.parametrize("mode", [INNER, CDIST, CORR])
def test_grouped_mixed_groups_in_one_launch(mode):
    """Nine groups of mixed sizes in one launch: every block must find its group by the block_begin search, and
    every group's cost entries (and nothing around them) are written."""
    for accumulate in (0, 1):
        _grouped_case(MIXED, mode, accumulate, seed=500 + 7 * accumulate + len(mode))


SPLITS = [1, 2, 3, 7, 48, 49, 200, 5]
LAYOUTS = ["gemm", "wide", "tma1", "direct", (100 + 3, 192), "gemm", (256, 128), "wide"]


@pytest.mark.parametrize("ntaps", range(1, 9))
def test_grouped_taps_per_group(ntaps):
    """1 to 8 taps in one group of 100 units with differing splits, ld_m, ld_n and n_affine (0, 1 or 2)."""
    taps = [(SPLITS[(i + ntaps) % 8], LAYOUTS[i], (i + ntaps) % 3, ("normal", "mean", "dead")[i % 3])
            for i in range(ntaps)]
    for k, mode in enumerate((INNER, CDIST, CORR)):
        _grouped_case([(100, 28, taps)], mode, (k + ntaps) % 2, seed=900 + 10 * ntaps + k)


@pytest.mark.parametrize("n,layout", [(40, "gemm"), (100, "gemm"), (200, "gemm"), (64, "direct"), (128, "direct"),
                                      (100, "tma1"), (128, "tma1"), (129, "tma2"), (600, "tma2")], ids=str)
def test_grouped_production_layouts(n, layout):
    """The partial layouts of GemmPlan (bn 64 / 128 / 256), DirectGramPlan and TmaGramPlan at cta_group 1 and 2."""
    for k, mode in enumerate((INNER, CDIST, CORR)):
        _grouped_case([(n, 0, [(3, layout, 1, "normal"), (4, layout, 0, "mean")])], mode, k % 2, seed=1300 + n + k)


@pytest.mark.parametrize("n_affine", [0, 1, 2])
@pytest.mark.parametrize("mode", [INNER, CDIST, CORR])
def test_grouped_derived_taps(mode, n_affine):
    """n_affine derived taps per contracted one, with s of both signs and exactly 0 and |t| up to ~300 |s|, on
    ordinary, large-mean and dead-unit inputs."""
    for kind in ("normal", "mean", "dead"):
        for accumulate in (0, 1):
            _grouped_case([(77, 11, [(3, "gemm", n_affine, kind)])], mode, accumulate,
                          seed=1700 + 10 * n_affine + len(kind) + accumulate)


def test_grouped_corr_dead_units_are_exactly_zero():
    """A unit without variance correlates with nothing: its row and column are exactly 0, derived taps included."""
    tap = _Tap(70, 3, "gemm", 2, "dead", 1900)
    g = _Group(70, 2, [tap], 0, 1901)
    _run_grouped([g], CORR, 0)
    c = g.cost[:, :70]
    dead_a, dead_b = tap.qa64 == 0, tap.qb64 == 0
    assert dead_a.any() and dead_b.any()
    assert (c[dead_a] == 0).all() and (c[:, dead_b] == 0).all()
    assert g.check(CORR) <= 1.0


# ------------------------------------------------------------------------------------------------ per-tap kernels


def _per_tap(M, Nn, splits, ld, mode, out_dtype, accumulate, sym_bn, seed):
    """plb_cross_finalize / plb_cross_finalize_corr on a synthetic tap; the cost is [M][ldc] inside a sentinel
    guard.  With sym_bn, only the entries of tiles touching the lower triangle may be written."""
    ops = _ops()
    n = max(M, Nn)
    tap = _Tap(n, splits, ld, 0, "mean" if mode == CORR else "normal", seed)
    ldc = Nn + 3
    flat, buf = _guarded(M * ldc, out_dtype, SENTINEL)
    cost = flat.view(M, ldc)
    gen = torch.Generator(device="cuda").manual_seed(seed + 1)
    cost[:, :Nn] = torch.randn(M, Nn, generator=gen, device="cuda", dtype=out_dtype) if accumulate else NAN
    old = cost[:, :Nn].double().clone()
    before_buf = buf.clone()
    if mode == CORR:
        ops.N.call("plb_cross_finalize_corr", flat.device, tap.partial.data_ptr(), splits, tap.ld_m, tap.ld_n, M, Nn,
                   tap.qa.data_ptr(), tap.qb.data_ptr(), tap.sa.data_ptr(), tap.sb.data_ptr(), tap.K, flat.data_ptr(),
                   ldc, int(accumulate))
    else:
        c32, c64 = (flat.data_ptr(), None) if out_dtype == torch.float32 else (None, flat.data_ptr())
        ops.N.call("plb_cross_finalize", flat.device, tap.partial.data_ptr(), splits, tap.ld_m, tap.ld_n, M, Nn,
                   tap.qa.data_ptr(), tap.qb.data_ptr(), _mode_code(mode), c32, c64, ldc, int(accumulate), sym_bn)
    torch.cuda.synchronize()
    i = torch.arange(M, device="cuda")[:, None]
    j = torch.arange(Nn, device="cuda")[None]
    live = ~((128 * (i // 128) + 127) < sym_bn * (j // sym_bn)) if sym_bn else torch.ones(M, Nn, dtype=torch.bool,
                                                                                           device="cuda")
    mask = torch.ones_like(buf, dtype=torch.bool)
    mask[GUARD:GUARD + M * ldc].view(M, ldc)[:, :Nn] = ~live
    bits = torch.int64 if out_dtype == torch.float64 else torch.int32
    assert torch.equal(buf[mask].view(bits), before_buf[mask].view(bits)), "written outside the live entries"
    v, b = tap.values(mode)[0]
    v, b = v[:M, :Nn], b[:M, :Nn]
    if out_dtype == torch.float64 and mode == INNER:
        b = E64 * tap.Pabs[:M, :Nn]  # the fp64 sum itself is stored
    ref = v + old if accumulate else v
    bar = b + (U if out_dtype == torch.float32 else 2.0 ** -52) * (v.abs() + old.abs() if accumulate else 0 * v)
    got = cost[:, :Nn].double()
    r = _note("per-tap", _ratio(torch.where(live, (got - ref).abs(), 0.0), torch.where(live, SLACK * bar, 1.0)))
    assert r <= 1.0, (M, Nn, splits, mode, out_dtype, accumulate, sym_bn, r)


@pytest.mark.parametrize("splits", [1, 2, 3, 47, 48, 49, 50, 200])
@pytest.mark.parametrize("mode", [INNER, CDIST])
def test_per_tap_finalize_stream_and_reduce(mode, splits):
    """plb_cross_finalize on either side of its switch from the streaming kernel (<= 48 splits) to the split-reduce
    kernel, fp32 and fp64 output, overwrite and accumulate, M != N."""
    for k, dtype in enumerate((torch.float32, torch.float64)):
        for accumulate in (0, 1):
            _per_tap(130, 97, splits, "gemm", mode, dtype, accumulate, 0, seed=2100 + splits + 10 * k + accumulate)


@pytest.mark.parametrize("sym_bn", [64, 128, 256])
@pytest.mark.parametrize("splits", [3, 49])
def test_per_tap_finalize_symmetric_mask(sym_bn, splits):
    """sym_bn: only the tiles a symmetric GEMM computed (touching the lower triangle) are written, the rest of the
    cost matrix stays bit-unchanged."""
    n = 300
    _per_tap(n, n, splits, (384, (n + sym_bn - 1) // sym_bn * sym_bn), INNER, torch.float32, 1, sym_bn,
             seed=2300 + sym_bn + splits)


@pytest.mark.parametrize("splits", [1, 2, 49, 200])
def test_per_tap_finalize_corr(splits):
    """plb_cross_finalize_corr, overwrite and accumulate, on large-mean rows."""
    for accumulate in (0, 1):
        _per_tap(70, 70, splits, "wide", CORR, torch.float32, accumulate, 0, seed=2500 + splits + accumulate)


# ------------------------------------------------------------------------------------------------ 2. derived vs contracted

COND_MU = [0.0, 0.5, 1.0, 2.0, 4.0, 16.0, 64.0]
COND_BETA = [0.0, 1.0, 4.0]
COND_SHAPE = (8, 96, 784)  # [outer, C, inner]: K = 6272, a 28x28 layer at batch 8


def _bn_side(mu_sigma, beta_gamma, neg_gamma, seed):
    """fp32 activations [outer, C, inner] whose units have mean mu and spread sigma with |mu| / sigma = mu_sigma, and
    the (s, t) of a BatchNorm calibrated on them (gamma in [0.5, 1.5], beta = +-beta_gamma gamma)."""
    outer, C, inner = COND_SHAPE
    gen = torch.Generator(device="cuda").manual_seed(seed)
    f64 = dict(dtype=torch.float64, device="cuda")
    # a small scale keeps the contracted tap's own value (added by the same launch) far below the derived one's error
    sigma = 2.0 ** -10 * (0.5 + 1.5 * torch.rand(C, generator=gen, **f64))
    sign = torch.randint(0, 2, (C,), generator=gen, device="cuda").double() * 2 - 1
    z = torch.randn(COND_SHAPE, generator=gen, **f64)
    x = ((mu_sigma * sigma * sign).view(1, C, 1) + sigma.view(1, C, 1) * z).float()
    xd = x.double()
    mean, var = xd.mean((0, 2)), xd.var((0, 2), unbiased=False)
    gamma = 0.5 + torch.rand(C, generator=gen, **f64)
    if neg_gamma:
        gamma[::3] *= -1.0
    beta = beta_gamma * gamma.abs() * (torch.randint(0, 2, (C,), generator=gen, device="cuda").double() * 2 - 1)
    s = gamma / var.sqrt()
    t = beta - mean * s
    return x, s, t, (mean, var, gamma, beta)


def _tma_tap(x, y):
    """TmaGramPlan on (x, y) with all four moment buffers; returns the plan and [qa, qb, sa, sb]."""
    ops = _ops()
    outer, C, inner = x.shape
    plan = ops.TmaGramPlan(C, outer, inner, x.device)
    q = torch.zeros(4, C, dtype=torch.float64, device="cuda")
    plan.run(x, y, 1, q[0], q[1], q[2], q[3])
    return plan, q


def _epilogue(plan, q, K, mode, affine=None):
    """The grouped epilogue of one tap (n_affine = 1 with ``affine``), overwriting an fp32 cost matrix."""
    ops = _ops()
    C = plan.M
    cost = torch.full((C, C), NAN, device="cuda")
    entry = ops.N.FinalizeTap(plan.partial.data_ptr(), q[0].data_ptr(), q[1].data_ptr(), q[2].data_ptr(),
                              q[3].data_ptr(), plan.ld_m, plan.ld_n, K, plan.splits, 0 if affine is None else 1,
                              ops.N.ptr(affine))
    arena = ops.TableArena("cuda")
    taps_t = arena.put(bytes(entry))
    groups_t = arena.put(bytes(ops.N.FinalizeGroup(cost.data_ptr(), C, C, 0, 1, 0)))
    ops.N.call("plb_cross_finalize_grouped", cost.device, taps_t.data_ptr(), groups_t.data_ptr(), 1,
               ops.finalize_grouped_blocks(C), _mode_code(mode), 0)
    torch.cuda.synchronize()  # before the table arena goes
    return cost


def _stat_ratio(mode, out, G64, A, mom, K):
    """Ratio of one tap's statistic to the contracted route's bar (tests/test_gram_gpu.py), 1 = at the bar."""
    if mode == INNER:
        return _ratio((out.double() - G64).abs(), A) / TOL
    if mode == CDIST:
        return _cdist_ratio(out, G64, A, mom) / TOL
    return _corr_ratio(out, G64, A, mom, K) / TOL


COND_CASES = [(mu, bg, False) for mu in COND_MU for bg in COND_BETA] + [(4.0, 1.0, True), (0.0, 0.0, True)]


@pytest.mark.parametrize("mu_sigma,beta_gamma,neg_gamma", COND_CASES, ids=str)
def test_derived_batchnorm_tap_conditioning(mu_sigma, beta_gamma, neg_gamma):
    """The derived statistic of a BatchNorm tap against the contracted one, both against fp64 on x' = s x + t.  The
    contracted route always meets its bar; the derived route must meet the same bar wherever BN_AFFINE_MAX_GROWTH
    admits the derivation."""
    AM = _am()
    K = COND_SHAPE[0] * COND_SHAPE[2]
    seed = 3000 + int(16 * mu_sigma) + 7 * int(beta_gamma) + 500 * neg_gamma
    x, s_a, t_a, st_a = _bn_side(mu_sigma, beta_gamma, neg_gamma, seed)
    y, s_b, t_b, st_b = _bn_side(mu_sigma, beta_gamma, neg_gamma, seed + 1)
    growth = AM.affine_growth(st_a[0], st_a[1], 0.0, st_a[2], st_a[3]) * \
        AM.affine_growth(st_b[0], st_b[1], 0.0, st_b[2], st_b[3])
    admitted = growth <= AM.BN_AFFINE_MAX_GROWTH
    affine = _guarded64(torch.cat([s_a, t_a, s_b, t_b]))
    xp64 = s_a.view(1, -1, 1) * x.double() + t_a.view(1, -1, 1)
    yp64 = s_b.view(1, -1, 1) * y.double() + t_b.view(1, -1, 1)
    G64, A, mom = _reference(xp64, yp64)
    plan, q = _tma_tap(x, y)
    plan_c, q_c = _tma_tap(xp64.float(), yp64.float())
    for mode in (INNER, CDIST, CORR):
        base = _epilogue(plan, q, K, mode)
        both = _epilogue(plan, q, K, mode, affine)
        derived = (both.double() - base.double()).float()  # the launch adds the tap in front's own value first
        contracted = _epilogue(plan_c, q_c, K, mode)
        rd = _stat_ratio(mode, derived, G64, A, mom, K)
        rc = _stat_ratio(mode, contracted, G64, A, mom, K)
        COND_TABLE.append((mu_sigma, beta_gamma, neg_gamma, mode, growth, rd, rc, admitted))
        print(f"\nmu/sigma {mu_sigma:g} beta/gamma {beta_gamma:g} gamma<0 {neg_gamma} {mode}: growth {growth:.4g} "
              f"derived {rd:.3g} contracted {rc:.3g} ({'derived' if admitted else 'contracted'} in activation_matching)")
        assert rc <= 1.0, (mode, rc)
        if admitted:
            assert rd <= 1.0, (mode, growth, rd)


# ------------------------------------------------------------------------------------------------ 4. end to end

E2E_BATCHES = 3


def _calibrated_tinynet_pair():
    """A tinynet pair whose BatchNorm running statistics are the cumulative averages over the calibration batches
    (train mode, momentum=None), as a trained network's are on in-distribution data: the convolutions behind a
    ReLU then produce outputs with |mean| of a few spreads, and the BatchNorm normalises that away."""
    from oracle import tinynet

    m1, m2 = tinynet.make_pair(12, 10)
    loader = tinynet.make_loader(E2E_BATCHES, 8, 16, seed=11)
    for m in (m1, m2):
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.reset_running_stats()
                mod.momentum = None
        m.train()
        with torch.no_grad():
            for x, _ in loader:
                m(x)
        m.eval()
    return m1, m2, loader


def _cross64(mode):
    """fp64 cross statistic of two activations along axis a (the reference's movedim + reshape)."""
    def cross(x, y, a):
        X = x.movedim(a, 0).reshape(x.shape[a], -1).double()
        Y = y.movedim(a, 0).reshape(y.shape[a], -1).double()
        if mode == INNER:
            return X @ Y.T
        if mode == CDIST:
            return -torch.cdist(X, Y)
        Xc, Yc = X - X.mean(1, keepdim=True), Y - Y.mean(1, keepdim=True)
        na, nb = Xc.norm(dim=1), Yc.norm(dim=1)
        C = (Xc @ Yc.T) / (na[:, None] * nb[None]).clamp_min(1e-300)
        return torch.where((na[:, None] > 0) & (nb[None] > 0), C, 0.0)
    return cross


def _bn_taps(spec, m1, m2):
    """{fx node name: (bn_a, bn_b)} of the tapped BatchNorm outputs."""
    out = {}
    for pg in spec.values():
        for ax in pg.node:
            name = ax.key
            for mod_name, mod in m1.named_modules():
                if isinstance(mod, torch.nn.BatchNorm2d) and mod_name.replace(".", "_") == name:
                    out[name] = (mod, m2.get_submodule(mod_name))
    return out


# largest cost error / max|cost| against fp64, measured on a B200: derived 2.0e-6 / 5.7e-7 / 6.9e-6 (inner / cdist /
# corr), contracted 2.1e-6 / 6.1e-7 / 6.9e-6; every BatchNorm tap derived, without the bound: 6.6e-6 / 1.2e-6 / 1.4e-5
E2E_BAR = {INNER: 4e-6, CDIST: 1e-6, CORR: 1e-5}


@pytest.mark.parametrize("mode", [INNER, CDIST, CORR])
def test_calibrated_batchnorm_taps_end_to_end(mode, monkeypatch):
    """activation_matching on a calibrated tinynet pair with BN_AFFINE on and off (and with no bound) against an fp64 run of the same
    models: both routes meet the same cost bar, the permutations are the fp64 costs' assignment (or objective-equal),
    and exactly the BatchNorm taps BN_AFFINE_MAX_GROWTH admits are derived (one Gram launch less each per batch)."""
    import copy

    from test_methods_gpu import assert_perm_or_objective

    AM = _am()
    P = __import__("pleas_merging_b200")
    from pleas_merging_b200 import _native

    m1, m2, loader = _calibrated_tinynet_pair()
    spec = P.get_permutation_spec(m1, ((1, 3, 16, 16),))
    bn_taps = _bn_taps(spec, m1, m2)
    admitted = [name for name, (a, b) in bn_taps.items() if AM._bn_derivable(a, b)]
    assert 0 < len(admitted) < len(bn_taps), (admitted, list(bn_taps))
    fn = {INNER: P.cross_features_inner_product, CDIST: P.cross_features_cdist,
          CORR: P.cross_features_correlation}[mode]
    d1, d2 = copy.deepcopy(m1).double().cuda(), copy.deepcopy(m2).double().cuda()
    axes = [ax for pg in spec.values() for ax in pg.node]
    gm = AM.build_cross_module(d1, d2, axes, _cross64(mode))
    ref = AM.compute_matching_costs(spec, gm, [(x.double(), 0) for x, _ in loader], E2E_BATCHES, accumulate="sum")
    g1, g2 = m1.cuda(), m2.cuda()
    runs = {}
    for label, flag, bound in (("derived", True, None), ("contracted", False, None), ("ungated", True, math.inf)):
        monkeypatch.setattr(AM, "BN_AFFINE", flag)
        if bound is not None:
            monkeypatch.setattr(AM, "BN_AFFINE_MAX_GROWTH", bound)
        AM.clear_caches()
        _native.LAUNCH_COUNTS.clear()
        perm, costs = P.activation_matching(spec, g1, g2, loader, E2E_BATCHES, cross_features=fn, output_costs=True,
                                            accumulate="sum", use_cuda_graph=False)
        grams = sum(_native.LAUNCH_COUNTS[k] for k in ("plb_gram_tma", "plb_pack_split_pair", "plb_pack_split_pair_sums"))
        errs = {k: float((costs[k].double() - ref[k]).abs().max()) / float(ref[k].abs().max()) for k in spec}
        runs[label] = (perm, grams, max(errs.values()))
    AM.clear_caches()
    print(f"\n{mode}: BatchNorm taps derived {len(admitted)} of {len(bn_taps)} ({', '.join(admitted)}); largest cost "
          "error / max|cost| against fp64: " + ", ".join(f"{k} {v[2]:.3g}" for k, v in runs.items()))
    assert runs["contracted"][1] - runs["derived"][1] == E2E_BATCHES * len(admitted)
    assert runs["contracted"][1] - runs["ungated"][1] == E2E_BATCHES * len(bn_taps)
    for label in ("derived", "contracted"):
        perm, _, err = runs[label]
        assert err <= E2E_BAR[mode], (label, err)
        for k in spec:
            assert_perm_or_objective(perm[k].numpy(), _assignment(ref[k]), ref[k].cpu().numpy(), f"{label} {k}")


def _assignment(cost):
    """The maximising assignment of an fp64 cost matrix (SciPy)."""
    from scipy.optimize import linear_sum_assignment

    _, col = linear_sum_assignment(cost.cpu().numpy(), maximize=True)
    return col


def test_refresh_refuses_statistics_the_bound_no_longer_admits():
    """BatchNorm statistics that change in place after the calibration graph was built keep the runner's fingerprint:
    a derived tap they no longer admit makes refresh_affines raise on a runner used directly, and activation_matching
    drops its cached runner and contracts that tap."""
    from oracle import tinynet

    AM = _am()
    P = __import__("pleas_merging_b200")
    from pleas_merging_b200 import _native

    m1, m2 = tinynet.make_pair(12, 10)
    g1, g2 = m1.cuda(), m2.cuda()
    spec = P.get_permutation_spec(m1, ((1, 3, 16, 16),))
    loader = tinynet.make_loader(2, 8, 16, seed=7)
    bn_a, bn_b = g1.layer1[0].bn2, g2.layer1[0].bn2
    assert AM._bn_derivable(bn_a, bn_b)

    def grams():
        return sum(_native.LAUNCH_COUNTS[k] for k in ("plb_gram_tma", "plb_pack_split_pair", "plb_pack_split_pair_sums"))

    AM.clear_caches()
    try:
        _native.LAUNCH_COUNTS.clear()
        P.activation_matching(spec, g1, g2, loader, 2, accumulate="sum", use_cuda_graph=False)
        first = grams()
        runner = next(iter(AM._RUNNER_CACHE.values()))[0]
        with torch.no_grad():
            bn_a.running_mean.add_(10.0 * bn_a.running_var.sqrt())  # |mean| / spread ~ 10: refused
        assert not AM._bn_derivable(bn_a, bn_b)
        with pytest.raises(RuntimeError, match="no longer admit"):
            runner.acc.refresh_affines()
        _native.LAUNCH_COUNTS.clear()
        _, costs = P.activation_matching(spec, g1, g2, loader, 2, output_costs=True, accumulate="sum",
                                         use_cuda_graph=False)
        assert next(iter(AM._RUNNER_CACHE.values()))[0] is not runner
        assert grams() == first + 2  # the layer1.0.bn2 tap is contracted in both batches
        AM.clear_caches()
        with pytest.MonkeyPatch.context() as mp:
            mp.setattr(AM, "BN_AFFINE", False)
            _, want = P.activation_matching(spec, g1, g2, loader, 2, output_costs=True, accumulate="sum",
                                            use_cuda_graph=False)
        for k in spec:  # the other BatchNorm taps are still derived: equal to the contracted ones within 1e-5
            assert float((costs[k] - want[k]).abs().max()) <= 1e-5 * float(want[k].abs().max()), k
    finally:
        AM.clear_caches()
