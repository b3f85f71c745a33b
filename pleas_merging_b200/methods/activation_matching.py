"""Activation matching on B200 (drop-in for pleas/methods/activation_matching.py).

Same public surface as the reference — ``cross_features_inner_product``,
``cross_features_cdist``, ``build_cross_module``, ``compute_matching_costs``,
``activation_matching`` — with the arithmetic moved into the library's kernels:

* every tap is one pass over the two activations (pack.cu: hi/lo split into tcgen05 operand
  order + row norms, no transposed copy), one 3xTF32 tcgen05 GEMM (gemm.cu) and one fused
  epilogue (finalize.cu) that applies ``-cdist``/inner product and adds straight into the tap's
  permutation-group cost matrix;
* all groups' assignment problems are solved in ONE launch of the GPU LAP kernel (lap.cu),
  bit-identical to SciPy's answer, with a single D2H copy of the permutations at the end.

``accumulate`` selects the batch semantics (SURVEY.md finding F1): ``"reference"`` (default)
reproduces the reference exactly — its membership test at activation_matching.py:124 compares
a tuple with ``Axis`` keys, so every batch overwrites and only the last processed batch
counts; ``"sum"`` is the paper-intended sum over batches.
"""
import itertools
import operator
import os
from collections.abc import Collection

import torch
import torch.fx
from torch.nn import Module

from .. import conv, ops
from ..core.solvers import b200_solve_lsa, solve_lsa_batched
from ..core.utils import Axis, Permutation, PermutationSpec
from ..graphs import GraphedStep
from ..parallel import BatchSharder, combine_costs_, device_prefetch


# ------------------------------------------------------------------ plug-compatible operators

def cross_features_inner_product(x, y, a: int):
    """[x.shape[a], y.shape[a]] Gram matrix over all other axes (reference :14-28)."""
    return ops.cross_statistic(x, y, a, ops.MODE_INNER)


def cross_features_cdist(x, y, a: int):
    """Negative Euclidean distance between the axis-``a`` slices (reference :31-46)."""
    return ops.cross_statistic(x, y, a, ops.MODE_NEG_CDIST)


def cross_features_correlation(x, y, a: int):
    """Pearson correlation between the axis-``a`` slices of x and y over all other axes — the third
    statistic BASELINE.json's north_star names (not in the reference, which ships the two siblings above):
    built from the cross-Gram, the per-unit sums and sums of squares the fused kernel accumulates in the
    same pass.  A unit without variance correlates with nothing (0, where numpy.corrcoef gives NaN)."""
    return ops.cross_statistic(x, y, a, ops.MODE_CORR)


_FUSED_MODES = {cross_features_inner_product: ops.MODE_INNER, cross_features_cdist: ops.MODE_NEG_CDIST,
                cross_features_correlation: ops.MODE_CORR}


# ------------------------------------------------------------------ dual-model graph

def _tap_axes(axes: Collection) -> dict:
    taps = {}
    for ax in axes:
        taps.setdefault(ax.key, set()).add(ax.axis)
    return {k: sorted(v) for k, v in taps.items()}


_INPLACE_FUNCTIONS = {operator.iadd, operator.isub, operator.imul, operator.itruediv, torch.relu_}


def _mutates_inputs(node, root):
    """Conservative test for fx nodes that may overwrite one of their inputs in place."""
    if node.op == "call_module":
        return bool(getattr(root.get_submodule(node.target), "inplace", False))
    if node.op == "call_method":
        return node.target.endswith("_") and not node.target.endswith("__")
    if node.op == "call_function":
        return node.target in _INPLACE_FUNCTIONS or bool(node.kwargs.get("inplace", False)) \
            or getattr(node.target, "__name__", "").endswith("_")
    return False


_CONV_PAIRS = {}
_conv_ids = itertools.count()


def _conv_pair_dispatch(pair_id: int, xa, xb):
    """fx ``call_function`` target: the same convolution layer of both models in one launch of the library's
    3xTF32 tcgen05 kernel (conv.ConvPair; falls back to the modules for inputs it does not cover)."""
    return _CONV_PAIRS[pair_id](xa, xb)


def _dual_graph(model1: Module, model2: Module, axes: Collection, emit, emit_sync=None, conv_pairs=None,
                emit_affine=None, on_layer=None):
    """Runs both models side by side in one fx graph (model2 must trace to model1's graph, as
    in the reference, :68).  After every tapped node ``emit(graph, name, axis, node_a, node_b)``
    inserts the tap consumer right behind its producers — torchvision's in-place ReLU
    overwrites the preceding tap's storage, so consumers must not be deferred.  ``emit_sync(graph)``
    (optional) is inserted before every node that may mutate an input: a consumer that reads taps
    asynchronously gets the chance to finish first.  ``conv_pairs`` (a list, optional): eligible Conv2d layers are
    not called as modules but pairwise through ``_conv_pair_dispatch``; the ids registered in ``_CONV_PAIRS`` are
    appended to the list for the caller to release.  ``emit_affine(node, axis, model1, model2)`` (optional) may claim a
    tap as a per-unit affine image of an earlier tap (returns True): no consumer is inserted for it.
    ``on_layer(graph, module_name, in_a, in_b, out_a, out_b)`` (optional) is called behind every Conv2d / Linear
    ``call_module`` node (PLeaS captures the trained layers' inputs and outputs this way)."""
    traced = torch.fx.symbolic_trace(model1)
    taps = _tap_axes(axes)
    g = torch.fx.Graph()
    env = ({}, {})
    emitted = {}
    out_a = out_b = None
    fused = {}  # BatchNorm / ReLU node -> (value_a, value_b) written by the convolution launch in front (None: never stored)
    for node in traced.graph.nodes:
        if node in fused:
            vals = fused[node]
            env[0][node], env[1][node] = vals if vals is not None else (None, None)
            for a in taps.get(node.name, ()):
                if emit_affine is not None and emit_affine(node, a, model1, model2):
                    emitted[node.name, a] = None
                else:  # _conv_fusion only leaves taps here that a value exists for
                    emitted[node.name, a] = emit(g, node.name, a, env[0][node], env[1][node])
            continue
        if node.op == "placeholder":
            ph = g.node_copy(node)
            env[0][node] = env[1][node] = ph
            continue
        if node.op == "output":
            out_a = torch.fx.node.map_arg(node.args[0], lambda n: env[0][n])
            out_b = torch.fx.node.map_arg(node.args[0], lambda n: env[1][n])
            continue
        if emit_sync is not None and _mutates_inputs(node, traced):
            emit_sync(g)
        pair = _conv_pair_for(node, model1, model2) if conv_pairs is not None else None
        if pair is not None:
            plan = _conv_fusion(node, model1, model2, taps, emit_affine) if CONV_BN_FUSION else None
            if plan is not None:
                bn_node, relu_node, bns = plan
                pair.bns, pair.relu = bns, relu_node is not None
            pid = next(_conv_ids)
            _CONV_PAIRS[pid] = pair
            conv_pairs.append(pid)
            both = g.call_function(_conv_pair_dispatch, (pid, env[0][node.args[0]], env[1][node.args[0]]))
            env[0][node] = g.call_function(operator.getitem, (both, 0))
            env[1][node] = g.call_function(operator.getitem, (both, 1))
            if on_layer is not None:
                on_layer(g, node.target, env[0][node.args[0]], env[1][node.args[0]], env[0][node], env[1][node])
            if plan is not None:
                second = (g.call_function(operator.getitem, (both, 2)), g.call_function(operator.getitem, (both, 3)))
                if relu_node is not None:
                    fused[bn_node], fused[relu_node] = None, second
                else:
                    fused[bn_node] = second
            for a in taps.get(node.name, ()):
                emitted[node.name, a] = emit(g, node.name, a, env[0][node], env[1][node])
            continue
        for side in (0, 1):
            new = g.node_copy(node, lambda n, side=side: env[side][n])
            if node.op in ("call_module", "get_attr"):
                new.target = f"{side}.{node.target}"
            env[side][node] = new
        if on_layer is not None and node.op == "call_module" and len(node.args) >= 1 and \
                isinstance(node.args[0], torch.fx.Node) and \
                isinstance(traced.get_submodule(node.target), (torch.nn.Conv2d, torch.nn.Linear)):
            on_layer(g, node.target, env[0][node.args[0]], env[1][node.args[0]], env[0][node], env[1][node])
        for a in taps.get(node.name, ()):
            if emit_affine is not None and emit_affine(node, a, model1, model2):
                emitted[node.name, a] = None
                continue
            emitted[node.name, a] = emit(g, node.name, a, env[0][node], env[1][node])
    g.output(([out_a, out_b], emitted))
    gm = torch.fx.GraphModule(torch.nn.ModuleList([model1, model2]), g)
    gm.graph.lint()
    return gm


# conv -> eval-mode BatchNorm (-> ReLU) chains of the source models run as ONE launch of the convolution kernel with
# two outputs (plb_conv2d_affine_forward) when the BatchNorm's own tap, if any, is derived from the convolution's
# (CrossAccumulator.emit_affine) — three passes over the activation less.  PLB_CONV_BN_FUSION=0 keeps the modules.
CONV_BN_FUSION = os.environ.get("PLB_CONV_BN_FUSION", "1") == "1"


def _is_relu_of(node, src, model1, model2):
    if node.kwargs and set(node.kwargs) - {"inplace"}:
        return False
    if node.op == "call_module":
        try:
            ms = (model1.get_submodule(node.target), model2.get_submodule(node.target))
        except AttributeError:
            return False
        return all(type(m) is torch.nn.ReLU and not m._forward_hooks and not m._forward_pre_hooks for m in ms) and \
            tuple(node.args) == (src,)
    if node.op == "call_function":
        return node.target in (torch.relu, torch.relu_, torch.nn.functional.relu) and tuple(node.args) == (src,)
    return False


def _conv_fusion(node, model1, model2, taps, emit_affine):
    """(bn_node, relu_node or None, (bn_a, bn_b)) when the convolution ``node`` feeds exactly one foldable BatchNorm
    whose taps can all be derived from the convolution's tap, else None."""
    if len(node.users) != 1:
        return None
    bn = next(iter(node.users))
    if bn.op != "call_module" or tuple(bn.args) != (node,) or bn.kwargs:
        return None
    try:
        bns = (model1.get_submodule(bn.target), model2.get_submodule(bn.target))
    except AttributeError:
        return None
    if not all(conv.bn_foldable(m) and not m._forward_hooks and not m._forward_pre_hooks for m in bns):
        return None
    if bns[0].num_features != bns[1].num_features:
        return None
    for a in taps.get(bn.name, ()):  # a tapped BatchNorm output must be derivable: it is never read
        if emit_affine is None or not emit_affine(bn, a, model1, model2, check_only=True):
            return None
    relu = None
    if len(bn.users) == 1:
        cand = next(iter(bn.users))
        if _is_relu_of(cand, bn, model1, model2):
            relu = cand
    return bn, relu, bns


def _conv_pair_for(node, model1, model2):
    """ConvPair for an fx ``call_module`` node that is the same eligible Conv2d in both models, else None."""
    if node.op != "call_module" or len(node.args) != 1 or node.kwargs:
        return None
    try:
        ma, mb = model1.get_submodule(node.target), model2.get_submodule(node.target)
    except AttributeError:
        return None
    if not (conv.eligible(ma) and conv.eligible(mb)) or ma._forward_hooks or mb._forward_hooks or \
            ma._forward_pre_hooks or mb._forward_pre_hooks:
        return None
    pair = conv.ConvPair(ma, mb)
    return pair if pair.same_geometry() else None


def _release_conv_pairs(ids):
    for pid in ids:
        _CONV_PAIRS.pop(pid, None)


def build_cross_module(model1: Module, model2: Module, axes: Collection, cross_features):
    """GraphModule returning ``([out1, out2], {(node_name, axis): cross_features(a, b, axis)})``
    (reference :49-100).  On CUDA models the eligible convolutions run pairwise on the library kernel, exactly
    as in the fused loop, so both paths see the same activations."""
    import weakref

    on_gpu = all(p.is_cuda for p in itertools.chain(model1.parameters(), model2.parameters()))
    pairs = [] if (conv.ENABLED and on_gpu) else None
    gm = _dual_graph(model1, model2, axes,
                     lambda g, name, a, na, nb: g.call_function(cross_features, (na, nb, a)), conv_pairs=pairs)
    if pairs:
        weakref.finalize(gm, _release_conv_pairs, pairs)
    return gm


# ------------------------------------------------------------------ fused accumulation

_SINKS = {}
_sink_ids = itertools.count()
_DEBUG_TIMES = {}


class _timed:
    """PLB_DEBUG_TIMING=1: accumulates host wall time of the set-up paths."""

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if os.environ.get("PLB_DEBUG_TIMING") == "1":
            import time
            self.t0 = time.perf_counter()

    def __exit__(self, *exc):
        if os.environ.get("PLB_DEBUG_TIMING") == "1":
            import time
            _DEBUG_TIMES[self.name] = _DEBUG_TIMES.get(self.name, 0.0) + time.perf_counter() - self.t0


def _tap_dispatch(sink_id: int, tap_id: int, xa, xb):
    """fx ``call_function`` target of the fused path (a plain def so codegen can name it)."""
    _SINKS[sink_id].tap(tap_id, xa, xb)
    return None


def _sync_dispatch(sink_id: int):
    """fx ``call_function`` target: the main stream waits for the packs still reading taps."""
    _SINKS[sink_id].sync_packs()
    return None


class _Arena:
    """Staging memory for the large taps: a ring of ``slots`` arenas, each holding the packed hi/lo
    planes of both operands and the K-split partial tiles of one tap.  With the pack and GEMM
    streams decoupled, tap t+1 is packed into the next slot while tap t is still being multiplied.
    Buffers that are outgrown are kept alive: CUDA graphs captured against them stay valid."""

    def __init__(self, device, slots=1):
        self.device, self.slots = device, slots
        self.plane_floats = 0
        self.partial_floats = 0
        self.version = 0
        self.buf = [None] * slots
        self.partial = [None] * slots
        self._retired = []

    def ensure(self, plane_floats, partial_floats):
        if plane_floats > self.plane_floats:
            self._retired.append(self.buf)
            self.plane_floats = int(plane_floats * 1.25)
            self.buf = [torch.empty(4, self.plane_floats, dtype=torch.float32, device=self.device)
                        for _ in range(self.slots)]
            self.version += 1
        if partial_floats > self.partial_floats:
            self._retired.append(self.partial)
            self.partial_floats = int(partial_floats * 1.25)
            self.partial = [torch.empty(self.partial_floats, dtype=torch.float32, device=self.device)
                            for _ in range(self.slots)]
            self.version += 1


class _View:
    """Planes-like view into the arena."""

    def __init__(self, hi, lo, rows, row_groups, k_blocks):
        self.hi, self.lo, self.rows, self.row_groups, self.k_blocks = hi, lo, rows, row_groups, k_blocks


# Taps whose GEMM is below this many FLOPs are "small": a launch of their own is mostly prologue,
# pipeline ramp and tail (~19 us for ~4 us of work on a ResNet-50 pair), so their GEMMs are deferred
# to the end of the batch and run as one grouped persistent launch per tile width.
DEFER_FLOPS = float(os.environ.get("PLB_DEFER_FLOPS", "3e9"))
# Taps below this many FLOPs keep the packed path even when the TMA-fed kernel could read them in place
# (0: every eligible tap uses the fused kernel)
TMA_MIN_FLOPS = float(os.environ.get("PLB_TMA_MIN_FLOPS", "0"))
# pending K-split partial tiles that trigger a grouped epilogue launch (they should still be L2-resident)
FINALIZE_FLUSH_BYTES = int(float(os.environ.get("PLB_FINALIZE_FLUSH_MB", "1e9")) * 2 ** 20)


class _TapState:
    """Geometry, row-norm buffer and GEMM plan of one tap for one pair of activation shapes."""
    __slots__ = ("ra", "rb", "kb", "K", "q", "plan", "version", "pa", "pb", "deferred", "group", "slot", "direct",
                 "tap")


class _Tap:
    __slots__ = ("name", "axis", "group", "states", "affine", "aff_vec", "aff_key")


# Eval-mode BatchNorm taps are not contracted: per unit the layer is y = s x + t, so its cross statistic follows from
# the Gram, row sums and sums of squares of the tap in front of it (plb_cross_finalize_grouped, n_affine).  On a
# ResNet-50 pair that is 53 of the 174 taps.  PLB_BN_AFFINE=0 contracts every tap.
BN_AFFINE = os.environ.get("PLB_BN_AFFINE", "1") == "1"
# A derived tap inherits the conditioning of the tap in front.  Per unit, its error is the error of that tap's Gram
# and row moments (relative to |x|) times |s|: it grows like kappa = sqrt(1 + mean^2 / var) of the convolution output,
# while the contracted BatchNorm output is conditioned by its own mean and spread, kappa' = sqrt(1 + beta^2 / gamma^2).
# A BatchNorm tap is derived only while max(kappa / kappa') over model 1's units times the same over model 2's stays at
# or below this bound; above it the tap is contracted like any other, and the convolution in front of it runs unfused.
# Measured on a B200 (tests/test_finalize_gpu.py, RESULTS.md): at a product of 2.08 the derived statistic reaches 0.53
# of the contracted route's error bar, at 2.6 it is 1.4 times over it, and from there it grows like 0.6-0.8 times the
# product.  Random-init networks sit at 1; BatchNorm statistics calibrated on data reach 3 to 7 behind a ReLU.
BN_AFFINE_MAX_GROWTH = 2.0


def affine_growth(running_mean, running_var, eps, weight, bias):
    """max over units of kappa / kappa' of an eval-mode BatchNorm (see BN_AFFINE_MAX_GROWTH); a unit with gamma = 0
    outputs a constant, which the derivation reproduces exactly, and counts 0."""
    m, v = running_mean.detach().double(), running_var.detach().double()
    k2 = 1.0 + m * m / (v + eps)
    g2 = weight.detach().double() ** 2 if weight is not None else torch.ones_like(m)
    b2 = bias.detach().double() ** 2 if bias is not None else torch.zeros_like(m)
    r2 = torch.where(g2 > 0, k2 * g2 / (g2 + b2), torch.zeros_like(k2))
    return float(r2.max().sqrt())  # NaN statistics give NaN: never derived


def _bn_derivable(bn_a, bn_b):
    """True when the taps of this BatchNorm pair may be derived from the tap in front (BN_AFFINE_MAX_GROWTH)."""
    growth = affine_growth(bn_a.running_mean, bn_a.running_var, bn_a.eps, bn_a.weight, bn_a.bias) * \
        affine_growth(bn_b.running_mean, bn_b.running_var, bn_b.eps, bn_b.weight, bn_b.bias)
    return growth <= BN_AFFINE_MAX_GROWTH


def _bn_scale_shift(bn):
    """(s, t) in float64 with bn(x) = s x + t per channel (eval mode, running statistics)."""
    s = (bn.running_var.detach().double() + bn.eps).rsqrt()
    if bn.weight is not None:
        s = s * bn.weight.detach().double()
    t = -bn.running_mean.detach().double() * s
    if bn.bias is not None:
        t = t + bn.bias.detach().double()
    return s, t


def _bn_key(bn):
    ts = (bn.running_mean, bn.running_var, bn.weight, bn.bias)
    return tuple(None if x is None else (x.data_ptr(), x._version) for x in ts)


class CrossAccumulator:
    """Receives (activation_a, activation_b) at every tap, in graph order, and accumulates the
    chosen cross statistic into its permutation group's cost matrix."""

    def __init__(self, spec: PermutationSpec, mode: int, device, overlap=False):
        self.mode, self.device = mode, device
        # overlap=True (opt-in, PLB_OVERLAP=1): the statistics pipeline (HBM-bound packs, tensor-bound
        # GEMMs) runs on side streams and overlaps the models' forward kernels (FFMA-bound cuDNN
        # convolutions) on the main stream.  Packs get their own stream (the main stream only ever waits for packs, before an in-place
        # op overwrites a tap) and the GEMM + epilogue stream trails it through a ring of arenas.
        self.overlap = overlap
        self.s_pack = torch.cuda.Stream(device) if overlap else None
        self.s_gemm = torch.cuda.Stream(device) if overlap else None
        self._pack_events, self._live = [], []
        self._slot_free = {}   # arena slot -> event recorded when its last GEMM + epilogue finished
        self._next_slot = 0
        self.keys = list(spec.keys())
        sizes = [spec[k].size for k in self.keys]
        self.flat = torch.zeros(sum(n * n for n in sizes), dtype=torch.float32, device=device)
        self.costs, off = [], 0
        for n in sizes:
            self.costs.append(self.flat[off:off + n * n].view(n, n))
            off += n * n
        self.group_of = {}
        for gi, k in enumerate(self.keys):
            for ax in spec[k].node:
                self.group_of[ax.key, ax.axis] = gi
        self.taps = []
        self.tap_index = {}  # (node name, axis) -> index into self.taps
        self.arena = _Arena(device, slots=4 if overlap else 1)
        self._retired = []  # plans replaced by a rebind; captured graphs may still point at them
        self._pending = []  # deferred (small) taps of the batch in flight
        self._final = []    # taps whose epilogue joins the next grouped launch
        self._final_bytes = 0
        self._final_tables = {}
        self._last_final = None
        self._groups = {}   # tuple of deferred states -> GroupedGemm
        self.pool = ops.SlabPool(device)      # planes / partial tiles / row norms of the deferred taps
        self.tables = ops.TableArena(device)  # GEMM problem-table entries
        self.sink_id = next(_sink_ids)
        _SINKS[self.sink_id] = self

    def close(self):
        _SINKS.pop(self.sink_id, None)
        self.pool.release()

    def emit_sync(self, g):
        return g.call_function(_sync_dispatch, (self.sink_id,))

    def sync_packs(self):
        if self._pack_events:
            main = torch.cuda.current_stream(self.device)
            for ev in self._pack_events:
                main.wait_event(ev)
            self._pack_events = []

    def emit(self, g, name, axis, na, nb):
        t = _Tap()
        t.name, t.axis, t.group, t.states = name, axis, self.group_of[name, axis], {}
        t.affine, t.aff_vec, t.aff_key = [], None, None
        self.taps.append(t)
        self.tap_index[name, axis] = len(self.taps) - 1
        return g.call_function(_tap_dispatch, (self.sink_id, len(self.taps) - 1, na, nb))

    def emit_affine(self, node, axis, model1, model2, check_only=False):
        """Claims the tap of an eval-mode BatchNorm whose input is itself tapped (same axis, same permutation
        group): it becomes a derived tap of that one.  True when claimed.  ``check_only``: asks ahead, while the
        parent's own tap is still to be emitted."""
        if not BN_AFFINE or self.overlap or node.op != "call_module" or len(node.args) != 1 or node.kwargs or axis != 1:
            return False
        parent = node.args[0]
        if not isinstance(parent, torch.fx.Node):
            return False
        if (parent.name, axis) not in (self.group_of if check_only else self.tap_index):
            return False
        try:
            mods = (model1.get_submodule(node.target), model2.get_submodule(node.target))
        except AttributeError:
            return False
        for m in mods:
            if not isinstance(m, torch.nn.modules.batchnorm._BatchNorm) or m.training or \
                    not m.track_running_stats or m.running_mean is None or m.running_var is None:
                return False
        if self.group_of.get((node.name, axis)) != self.group_of.get((parent.name, axis)):
            return False
        n = self.costs[self.group_of[node.name, axis]].shape[0]
        if mods[0].num_features != n or mods[1].num_features != n:
            return False
        # an ill-conditioned derivation is refused: the tap is contracted, and _conv_fusion (which asks here first)
        # leaves the convolution in front unfused, since the BatchNorm output it would skip storing is now read
        if not _bn_derivable(*mods):
            return False
        if not check_only:
            self.taps[self.tap_index[parent.name, axis]].affine.append(mods)
        return True

    def affines_admitted(self):
        """True while every derived tap's BatchNorm pair still passes BN_AFFINE_MAX_GROWTH.  A derived tap cannot be
        switched to contraction in place (its BatchNorm output may not even be stored), so statistics that moved
        past the bound after the graph was built need a new graph."""
        return all(all(_bn_derivable(a, b) for a, b in t.affine) for t in self.taps
                   if t.affine and tuple((_bn_key(a), _bn_key(b)) for a, b in t.affine) != t.aff_key)

    def refresh_affines(self):
        """(Re)computes the derived taps' scale / shift vectors when the BatchNorm tensors changed (in place:
        captured graphs and epilogue tables keep pointing at the same buffer).  Raises when the new statistics no
        longer admit a derivation (affines_admitted)."""
        for t in self.taps:
            if not t.affine:
                continue
            key = tuple((_bn_key(a), _bn_key(b)) for a, b in t.affine)
            if key == t.aff_key:
                continue
            if not all(_bn_derivable(a, b) for a, b in t.affine):
                raise RuntimeError(f"tap {t.name}: the BatchNorm statistics behind it no longer admit a derived tap "
                                   "(BN_AFFINE_MAX_GROWTH); build a new CalibrationRunner")
            parts = []
            for a, b in t.affine:
                sa, ta = _bn_scale_shift(a)
                sb, tb = _bn_scale_shift(b)
                parts += [sa, ta, sb, tb]
            vec = torch.cat(parts).to(self.device)
            if t.aff_vec is None:
                t.aff_vec = vec.contiguous()
            else:
                t.aff_vec.copy_(vec)
            t.aff_key = key

    def begin_batch(self, reset_costs):
        self._pending, self._pack_events, self._live, self._final, self._final_bytes = [], [], [], [], 0
        self._slot_free, self._next_slot = {}, 0
        if reset_costs:
            self.flat.zero_()
        qs = [st.q for t in self.taps for st in t.states.values() if st.q is not None]
        if qs:
            torch._foreach_zero_(qs)

    def _prepare(self, t, xa, xb):
        oa, ra, ia = ops.as_rows_view(xa, t.axis)
        ob, rb, ib = ops.as_rows_view(xb, t.axis)
        if oa * ia != ob * ib:
            raise ValueError(f"tap {t.name}: contraction sizes differ between the two models")
        n = self.costs[t.group].shape[0]
        if (ra, rb) != (n, n):
            raise ValueError(f"tap {t.name}:{t.axis} has {ra}x{rb} units but its group has {n}")
        st = _TapState()
        st.tap = t
        st.ra, st.rb, st.K, st.kb = ra, rb, oa * ia, (oa * ia + 15) // 16
        # fp64 row norms live in the slab too (zeroed by begin_batch before the first use)
        # [qa | qb] sums of squares, [sa | sb] sums for the correlation statistic
        nq = {ops.MODE_INNER: 0, ops.MODE_NEG_CDIST: ra + rb, ops.MODE_CORR: 2 * (ra + rb)}[self.mode]
        if t.affine:  # derived taps are formed from the row sums as well
            nq = 2 * (ra + rb)
        st.q = self.pool.empty(2 * nq).view(torch.float64).zero_() if nq else None
        st.plan, st.version, st.group, st.slot = None, -1, t.group, None
        # narrow taps (C <= 128) are HBM-bound: the fused kernel reads the activations once, in place,
        # right behind their producer — no planes, nothing deferred
        fp32 = xa.dtype == torch.float32 and xb.dtype == torch.float32
        # TMA-fed fused kernel (any width): reads the activations in place, right behind their producer
        if (not self.overlap) and fp32 and ops.tma_gram_eligible(xa, xb, t.axis) and \
                2.0 * ra * rb * st.K >= TMA_MIN_FLOPS:
            st.direct, st.deferred, st.pa, st.pb, st.version = True, False, None, None, None
            st.plan = ops.TmaGramPlan(ra, oa, ia, self.device, pool=self.pool)
            return st
        st.direct = (not self.overlap) and fp32 and self.mode != ops.MODE_CORR and not t.affine and \
            ops.direct_gram_eligible(xa, xb, t.axis)
        if st.direct:
            st.deferred, st.pa, st.pb, st.version = False, None, None, None
            st.plan = ops.DirectGramPlan(ra, st.K, self.device, pool=self.pool)
            return st
        st.deferred = 2.0 * ra * rb * st.K < DEFER_FLOPS
        if st.deferred:  # own planes and partial tiles: they must survive until the end of the batch
            bn = ops.choose_bn(rb)
            m_tiles, n_tiles = (ra + 127) // 128, (rb + bn - 1) // bn
            splits = max(1, min(st.kb // 32, 16))
            st.pa = ops.Planes(ra, st.kb, self.device, pool=self.pool)
            st.pb = ops.Planes(rb, st.kb, self.device, pool=self.pool)
            st.plan = ops.GemmPlan(st.pa, st.pb, ra, rb, st.kb, splits=splits, pool=self.pool, tables=self.tables)
            st.plan.alg_flops = 2.0 * ra * rb * st.K
            st.version = None
        return st

    def _bind(self, st):
        """(Re)creates the tap's GEMM problem entry against the current arena."""
        rga, rgb = ops.row_groups_of(st.ra), ops.row_groups_of(st.rb)
        bn = ops.choose_bn(st.rb)
        m_tiles, n_tiles = (st.ra + 127) // 128, (st.rb + bn - 1) // bn
        splits = ops.choose_splits(m_tiles * n_tiles, st.kb, 128, bn)
        self.arena.ensure(max(rga, rgb) * st.kb * 128, splits * m_tiles * 128 * n_tiles * bn)
        if st.slot is None:  # taps run in the same order every batch, so a tap keeps its slot
            st.slot = self._next_slot
        b = self.arena.buf[st.slot]
        if st.plan is not None:
            self._retired.append((st.plan, st.pa, st.pb))
        st.pa = _View(b[0], b[1], st.ra, rga, st.kb)
        st.pb = _View(b[2], b[3], st.rb, rgb, st.kb)
        # own partial tiles (not the arena's): every tap's epilogue is deferred to ONE grouped launch at the end
        # of the batch, so its partials must survive until then
        st.plan = ops.GemmPlan(st.pa, st.pb, st.ra, st.rb, st.kb, splits=splits,
                               partial=self.pool.empty(splits * m_tiles * 128 * n_tiles * bn), tables=self.tables)
        st.plan.alg_flops = 2.0 * st.ra * st.rb * st.K
        st.version = self.arena.version

    def rebind_stale(self):
        """Binds every tap state against the final arena (outside any graph capture)."""
        for t in self.taps:
            for st in t.states.values():
                if not st.deferred and not st.direct and st.version != self.arena.version:
                    self._bind(st)
        if self._last_final:  # the epilogue table of the next (captured) batch exists before the capture starts
            self._final_table(self._last_final)

    def _state(self, idx, xa, xb):
        t = self.taps[idx]
        key = (tuple(xa.shape), tuple(xb.shape))
        st = t.states.get(key)
        if st is None:
            with _timed("prepare"):
                st = t.states[key] = self._prepare(t, xa, xb)
        if not st.deferred and not st.direct:
            if st.version != self.arena.version:
                with _timed("bind"):
                    self._bind(st)
            self._next_slot = (st.slot + 1) % self.arena.slots
        return t, st

    @staticmethod
    def _moments(st):
        """(qa, qb, sa, sb) views of the tap's fp64 row-moment buffer (None where the mode has none)."""
        if st.q is None:
            return None, None, None, None
        n = st.ra + st.rb
        qa, qb = st.q[:st.ra], st.q[st.ra:n]
        if st.q.numel() > n:
            return qa, qb, st.q[n:n + st.ra], st.q[n + st.ra:]
        return qa, qb, None, None

    def _pack(self, t, st, xa, xb):
        if xa.dtype != torch.float32:  # half / bf16 models: the statistics are computed in fp32
            xa = xa.float()
        if xb.dtype != torch.float32:
            xb = xb.float()
        qa, qb, sa, sb = self._moments(st)
        ops.pack_split_pair(xa, xb, t.axis, st.pa, st.pb, qa, qb, sa, sb)

    def _multiply(self, st):
        st.plan.run()
        self._multiply_epilogue(st)

    def tap(self, idx, xa, xb):
        t, st = self._state(idx, xa, xb)
        if st.direct:
            qa, qb, sa, sb = self._moments(st)
            if not xa.is_contiguous() or not xb.is_contiguous():  # same shape as a contiguous earlier batch
                xa, xb = xa.contiguous(), xb.contiguous()
            if sa is not None:
                st.plan.run(xa, xb, t.axis, qa, qb, sa, sb)
            else:
                st.plan.run(xa, xb, t.axis, qa, qb)
            self._multiply_epilogue(st)
            return
        if not self.overlap:
            self._pack(t, st, xa, xb)
            if st.deferred:
                self._pending.append(st)
            else:
                self._multiply(st)
            return
        main = torch.cuda.current_stream(self.device)
        ready = torch.cuda.Event()
        ready.record(main)
        self._live.append((xa, xb))  # the activations' memory must not be reused while a side stream reads it
        with torch.cuda.stream(self.s_pack):
            self.s_pack.wait_event(ready)
            if not st.deferred and st.slot in self._slot_free:
                self.s_pack.wait_event(self._slot_free[st.slot])  # the slot's previous tap is done with it
            self._pack(t, st, xa, xb)
            packed = torch.cuda.Event()
            packed.record(self.s_pack)
        self._pack_events.append(packed)
        if st.deferred:
            self._pending.append(st)
            return
        with torch.cuda.stream(self.s_gemm):
            self.s_gemm.wait_event(packed)
            self._multiply(st)
            free = torch.cuda.Event()
            free.record(self.s_gemm)
        self._slot_free[st.slot] = free

    def end_batch(self):
        """Runs the deferred small taps: one grouped GEMM launch per tile width, then their
        epilogues (in tap order, so the accumulation order is deterministic); joins the side streams."""
        if not self.overlap:
            return self._end_batch()
        main = torch.cuda.current_stream(self.device)
        packs_done = torch.cuda.Event()
        packs_done.record(self.s_pack)
        with torch.cuda.stream(self.s_gemm):
            self.s_gemm.wait_event(packs_done)
            self._end_batch()
            done = torch.cuda.Event()
            done.record(self.s_gemm)
        main.wait_event(done)
        self._pack_events, self._live, self._slot_free = [], [], {}

    def _end_batch(self):
        pending, self._pending = self._pending, []
        for bn in (64, 128, 256):
            sts = tuple(st for st in pending if st.plan.bn == bn)
            if not sts:
                continue
            grp = self._groups.get(sts)
            if grp is None:
                with _timed("group"):
                    grp = self._groups[sts] = ops.GroupedGemm([st.plan for st in sts], tables=self.tables)
            grp.run()
        for st in pending:
            self._multiply_epilogue(st)
        self._finalize_all()

    def _multiply_epilogue(self, st):
        """The tap's split-K reduction + statistic epilogue joins the batch's grouped launch (ONE per batch by
        default).  PLB_FINALIZE_FLUSH_MB flushes earlier, while the partial tiles are still in L2 — measured slower
        on a ResNet-50 pair: 28.3 ms/step with 38 launches (48 MB), 27.6 with 20 (96 MB), 26.3 with one, although
        that one reads its 2 GB of partials back from DRAM."""
        self._final.append(st)
        pl = st.plan
        self._final_bytes += 4 * pl.splits * pl.ld_m * pl.ld_n
        if self._final_bytes >= FINALIZE_FLUSH_BYTES:
            self._finalize_all()

    def _final_table(self, sts):
        """Device tables (taps in order per group) of the grouped epilogue for this list of tap states."""
        key = tuple((id(st), id(st.plan)) for st in sts)  # a rebind replaces the plan (new partial tiles)
        entry = self._final_tables.get(key)
        if entry is None:
            by_group = {}
            for st in sts:
                by_group.setdefault(st.group, []).append(st)
            taps_raw, groups_raw, blocks = bytearray(), bytearray(), 0
            ntaps = 0
            for gi in sorted(by_group):
                n = self.costs[gi].shape[0]
                members = by_group[gi]
                for st in members:
                    qa, qb, sa, sb = self._moments(st)
                    pl = st.plan
                    aff = st.tap.affine
                    if aff and st.tap.aff_vec is None:
                        self.refresh_affines()
                    taps_raw += bytes(ops.N.FinalizeTap(pl.partial.data_ptr(), ops.N.ptr(qa), ops.N.ptr(qb),
                                                        ops.N.ptr(sa), ops.N.ptr(sb), pl.ld_m, pl.ld_n, st.K,
                                                        pl.splits, len(aff), ops.N.ptr(st.tap.aff_vec) if aff else None))
                groups_raw += bytes(ops.N.FinalizeGroup(self.costs[gi].data_ptr(), self.costs[gi].stride(0), n, ntaps,
                                                        ntaps + len(members), blocks))
                ntaps += len(members)
                blocks += ops.finalize_grouped_blocks(n)
            entry = (self.tables.put(bytes(taps_raw)), self.tables.put(bytes(groups_raw)),
                     len(by_group), blocks, [(st, st.plan) for st in sts])  # keeps states / plans / buffers alive
            self._final_tables[key] = entry
        return entry

    def _finalize_all(self):
        """ONE launch for the epilogues of the pending taps (plb_cross_finalize_grouped): per permutation
        group the taps are reduced and added in tap order, each cost entry is touched once."""
        sts, self._final, self._final_bytes = self._final, [], 0
        if not sts:
            return
        self._last_final = sts
        taps_t, groups_t, ngroups, blocks, _ = self._final_table(sts)
        ops.N.call("plb_cross_finalize_grouped", self.device, taps_t.data_ptr(), groups_t.data_ptr(), ngroups, blocks,
                   self.mode, 1)


# ------------------------------------------------------------------ public API

def _model_device(model):
    p = next(iter(model.parameters()), None)
    if p is None or not p.is_cuda:
        raise RuntimeError("pleas_merging_b200 runs on a CUDA device: move both models to cuda first "
                           "(there is no CPU fallback)")
    return p.device


def compute_matching_costs(spec: PermutationSpec, gm_cross: Module, dataloader, num_batches,
                           accumulate="reference"):
    """Generic (un-fused) cost loop for a module built by ``build_cross_module`` with any
    ``cross_features`` callable (reference :103-136)."""
    if accumulate not in ("reference", "sum"):
        raise ValueError("accumulate must be 'reference' or 'sum'")
    device = _model_device(gm_cross)
    cross_sum = {}
    with torch.inference_mode():
        for (x, _), _ in zip(dataloader, range(num_batches)):
            _, cross = gm_cross(x.to(device, non_blocking=True))
            for ka, v in cross.items():
                k = Axis(*ka)
                if accumulate == "sum" and k in cross_sum:
                    cross_sum[k].add_(v)
                else:
                    cross_sum[k] = v
    costs = {}
    for key, pg in spec.items():
        present = [cross_sum[n] for n in pg.node if n in cross_sum]
        costs[key] = sum(present[1:], present[0].clone()) if present else 0
    return costs


class CalibrationRunner:
    """Streams calibration batches through the dual-model graph; the per-batch pipeline (two
    forwards + pack / GEMM / epilogue per tap) is replayed as a CUDA graph (graphs.GraphedStep)."""

    def __init__(self, spec, model1, model2, mode, accumulate="reference", use_cuda_graph=True, overlap=None):
        self.device = _model_device(model1)
        if overlap is None:
            # opt-in: the multi-stream pipeline saves ~5 % per batch on a ResNet-50 pair but its first
            # batch and graph capture cost ~0.35 s more, which only pays off beyond ~200 batches
            overlap = os.environ.get("PLB_OVERLAP", "0") == "1"
        self.acc = CrossAccumulator(spec, mode, self.device, overlap=overlap)
        axes = [ax for pg in spec.values() for ax in pg.node]
        self.conv_pairs = []
        self.gm = _dual_graph(model1, model2, axes, self.acc.emit, self.acc.emit_sync if overlap else None,
                              conv_pairs=self.conv_pairs if conv.ENABLED else None, emit_affine=self.acc.emit_affine)
        self.acc.refresh_affines()
        self.reset = accumulate == "reference"
        self.step = GraphedStep(self._eager, self.acc.rebind_stale, use_cuda_graph)

    def close(self):
        self.step.clear()
        self.acc.close()
        for pid in self.conv_pairs:
            _CONV_PAIRS.pop(pid, None)
        self.conv_pairs = []

    def refresh_weights(self):
        """Re-splits convolution weights that changed since they were packed (a CUDA-graph replay runs no
        Python: the packed planes it reads are brought up to date here, before the batches of a call)."""
        for pid in self.conv_pairs:
            _CONV_PAIRS[pid].refresh()
        self.acc.refresh_affines()

    def _eager(self, x):
        self.acc.begin_batch(reset_costs=self.reset)
        self.gm(x)
        self.acc.end_batch()

    def run(self, x):
        """One calibration batch (x on the models' device)."""
        self.step(x)


# The dual-model graph, the kernels' plans and the captured CUDA graph of a calibration step depend on the two
# modules, the spec and the batch shape only — not on the weights' values, which the replay reads in place.  The
# last runner is therefore kept for the next call with the same modules (sweeps over loaders / budgets, the
# warm-up call of a benchmark): it skips the fx trace, the eager first batch and the graph capture (~0.15 s for a
# ResNet-50 pair).  A fingerprint of every parameter / buffer address, shape and dtype and of the modules'
# training flags guards the reuse; PLB_RUNNER_CACHE=0 or clear_caches() switch it off / drop it.
_RUNNER_CACHE = {}
RUNNER_CACHE = os.environ.get("PLB_RUNNER_CACHE", "1") == "1"


def _model_fingerprint(model):
    fp = [(n, t.data_ptr(), tuple(t.shape), t.dtype) for n, t in itertools.chain(model.named_parameters(),
                                                                                 model.named_buffers())]
    return tuple(fp), tuple(m.training for m in model.modules())


def _spec_fingerprint(spec):
    return tuple((k.key, k.axis, pg.size, tuple(sorted((a.key, a.axis) for a in pg.node))) for k, pg in spec.items())


def clear_caches():
    """Drops the cached calibration runner (its CUDA graphs and staging memory) and the staging chunks kept
    for reuse."""
    for runner, _ in _RUNNER_CACHE.values():
        runner.close()
    _RUNNER_CACHE.clear()
    ops.SlabPool.trim()


def _get_runner(spec, model1, model2, mode, accumulate, use_cuda_graph):
    import weakref

    key = (id(model1), id(model2), mode, accumulate, bool(use_cuda_graph))
    fp = (_spec_fingerprint(spec), _model_fingerprint(model1), _model_fingerprint(model2))
    hit = _RUNNER_CACHE.get(key) if RUNNER_CACHE else None
    if hit is not None:
        runner, (refs, old_fp) = hit
        # BatchNorm statistics updated in place keep the fingerprint: a derived tap they no longer admit needs a new
        # graph, in which that tap is contracted
        if refs[0]() is model1 and refs[1]() is model2 and old_fp == fp and runner.acc.affines_admitted():
            runner.acc.flat.zero_()
            return runner
    clear_caches()  # at most one runner is kept: its graph pools hold several GB
    runner = CalibrationRunner(spec, model1, model2, mode, accumulate, use_cuda_graph)
    if RUNNER_CACHE:
        _RUNNER_CACHE[key] = (runner, ((weakref.ref(model1), weakref.ref(model2)), fp))
    return runner


def _fused_costs(spec, model1, model2, dataloader, num_batches, mode, accumulate, distributed=False,
                 use_cuda_graph=True):
    debug = os.environ.get("PLB_DEBUG_TIMING") == "1"
    if debug:
        import time
        torch.cuda.synchronize()
        marks = [("start", time.perf_counter())]
    runner = _get_runner(spec, model1, model2, mode, accumulate, use_cuda_graph)
    ok = False
    try:
        runner.refresh_weights()
        sharder = BatchSharder(dataloader, num_batches, *(() if distributed else (0, 1)))
        with torch.inference_mode():
            for i, x in device_prefetch(sharder, runner.device):
                runner.run(x)
                if debug and i < 3:
                    torch.cuda.synchronize()
                    marks.append((f"batch{i}", time.perf_counter()))
        acc = runner.acc
        combine_costs_(acc.flat, sharder, accumulate)
        out = {k: c.clone() for k, c in zip(acc.keys, acc.costs)}
        if debug:
            torch.cuda.synchronize()
            marks.append(("loop_end", time.perf_counter()))
            print("[plb timing] " + " ".join(f"{n}+{t - marks[0][1]:.3f}" for n, t in marks[1:]),
                  f"reserved {torch.cuda.memory_reserved() / 2**30:.1f} GiB",
                  "setup " + " ".join(f"{k}={v:.3f}s" for k, v in _DEBUG_TIMES.items()), flush=True)
            _DEBUG_TIMES.clear()
        ok = True
        return out
    finally:
        if not (ok and RUNNER_CACHE):  # a failed run may leave the runner half-way through a batch
            _RUNNER_CACHE.pop((id(model1), id(model2), mode, accumulate, bool(use_cuda_graph)), None)
            runner.close()


def activation_matching(
    spec: PermutationSpec,
    model1: Module,
    model2: Module,
    dataloader,
    num_batches=1000,
    cross_features=cross_features_cdist,
    lsa_solver=b200_solve_lsa,
    output_costs=False,
    *,
    accumulate="reference",
    distributed=False,
    use_cuda_graph=True,
) -> Permutation:
    """Permute model2's units to match model1's activations (reference :139-177).

    Returns ``{group key: CPU int64[n]}`` in spec order, plus the device fp32 ``[n, n]`` cost
    matrices when ``output_costs`` is set.  With the library's own ``cross_features`` /
    ``lsa_solver`` (the defaults) the fused kernels run; any other callable is honoured through
    the generic per-tap path.  ``distributed=True`` (inside an initialised torch.distributed
    job, every rank passing the SAME loader) deals the batches round-robin over the ranks and
    sums the cost matrices with one all-reduce; every rank returns the full result."""
    if accumulate not in ("reference", "sum"):
        raise ValueError("accumulate must be 'reference' or 'sum'")
    if cross_features in _FUSED_MODES:
        costs = _fused_costs(spec, model1, model2, dataloader, num_batches, _FUSED_MODES[cross_features], accumulate,
                             distributed, use_cuda_graph)
    else:
        if distributed:
            raise NotImplementedError("distributed=True needs the library's own cross_features operators")
        axes = [ax for pg in spec.values() for ax in pg.node]
        gm = build_cross_module(model1, model2, axes, cross_features)
        costs = compute_matching_costs(spec, gm, dataloader, num_batches, accumulate)
    if lsa_solver is b200_solve_lsa:
        if os.environ.get("PLB_DEBUG_TIMING") == "1":
            import time
            torch.cuda.synchronize()
            t0 = time.perf_counter()
        perm = dict(zip(costs.keys(), solve_lsa_batched(costs.values())))
        if os.environ.get("PLB_DEBUG_TIMING") == "1":
            print(f"[plb timing] batched LAP {time.perf_counter() - t0:.3f}s", flush=True)
    else:
        perm = {k: lsa_solver(v) for k, v in costs.items()}
    if output_costs:
        return perm, costs
    return perm


def check_multi_axis(spec):
    """True when some fx node contributes more than one axis to the spec (reference :180-194,
    restated with the evident intent: the reference never adds to its ``counter``)."""
    seen = set()
    for pg in spec.values():
        for ax in pg.node:
            if ax.key in seen:
                return True
            seen.add(ax.key)
    return False
