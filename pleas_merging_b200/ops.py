"""Tensor-level wrappers over the C ABI (include/pleas_b200.h).

PyTorch is plumbing here: it owns device memory and the current stream; every arithmetic
step is one of the library's sm_100a kernels.  Nothing in this module falls back to a CPU or
torch implementation.
"""
import ctypes
import os

import torch

from . import _native as N

MODE_INNER, MODE_NEG_CDIST, MODE_CORR = 0, 1, 2
NUM_SMS = 148  # B200; planning helpers ask the device (num_sms()) when one is present


def num_sms(device=None):
    """SM count of ``device`` (cached per ordinal); the B200 figure on a host without a GPU."""
    return N.sm_count(device) if torch.cuda.is_available() else NUM_SMS
# GEMM implementations behind plb_gemm_grouped:
#   "tcgen05"    persistent tcgen05 3xTF32 kernel with in-kernel promotion (product path)
#   "tcgen05_v1" one CTA per K chain, chains summed by the finalize kernel
#   "simt"       SIMT fp32 FMA cross-check kernel on the same planes (debugging only; still CUDA)
_GEMM_IMPL = os.environ.get("PLB_GEMM_IMPL", "tcgen05")
assert _GEMM_IMPL in ("tcgen05", "tcgen05_v1", "simt")
DIRECT_TIMER = None  # (start, end, algorithmic bytes, flops) per fused narrow-tap launch
PACK_TIMER = None  # set to a list by bench.py to collect (start, end, algorithmic bytes) per pack_split launch
GEMM_TIMER = None  # set to a list by bench.py to collect (start, end, flops, bn, n_problems) per GEMM launch


def _timer_events():
    """Two CUDA events for bracketing ONE launch on the current stream (bench instrumentation).  A short spin
    kernel is enqueued first so that the stream is still busy while the host submits the event, the launch and the
    second event: otherwise the first event completes at once and the measured interval includes the host's
    submission latency of the launch (~5-10 us from Python, 10 % of a 70 us kernel), which a CUDA-graph replay
    of the same launch never sees."""
    torch.cuda._sleep(60000)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    return e0, e1


def set_gemm_impl(name):
    global _GEMM_IMPL
    assert name in ("tcgen05", "tcgen05_v1", "simt")
    _GEMM_IMPL = name


def _impl_code(name):
    return {"tcgen05": 16 * MAX_CHAIN_KB, "tcgen05_v1": 0, "simt": 1}[name]


def _require_cuda_f32(t, what):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32):
        raise TypeError(f"{what}: expected a float32 CUDA tensor, got "
                        f"{type(t).__name__} {getattr(t, 'dtype', None)} on {getattr(t, 'device', None)}")


def row_groups_of(rows):
    """8-row groups of a packed operand.  Tight (no padding to the 128-row MMA tile): the GEMM
    producer copies only the groups that exist, so narrow operands (C = 64) cost their own bytes."""
    return (rows + 7) // 8


def plane_geometry(rows, K):
    """(row_groups, k_blocks, floats per plane) of the packed layout."""
    rg = row_groups_of(rows)
    kb = (K + 15) // 16
    return rg, kb, rg * kb * 128


class SlabPool:
    """Bump allocator over a few large device chunks.

    Every cudaMalloc is device-synchronous, so hundreds of per-tap ``torch.empty`` calls in the
    first calibration batch stall the host behind the queued forward kernels (measured: 1.4-2.4 s
    for a ResNet-50 pair).  A pool takes chunks of 0.5 GB and up (doubling), hands out 256-byte
    aligned float32 views, and on ``release()`` returns its chunks to a per-device free list that
    later pools reuse, so repeated calls allocate nothing.  A released chunk carries an event recorded
    on the releasing stream; whoever reuses it waits for that event first (side streams of the previous
    owner may still be reading it).  ``SlabPool.trim()`` hands the cached chunks back to PyTorch's
    allocator."""
    _free = {}  # device -> list of (float32 chunk, release event)

    def __init__(self, device):
        self.device = torch.device(device)
        self.chunks, self.used = [], 0
        self.next_floats = 1 << 27  # 0.5 GB

    def empty(self, nfloats):
        nfloats = max(int(nfloats), 1)
        need = (nfloats + 63) // 64 * 64
        if not self.chunks or self.used + need > self.chunks[-1].numel():
            free = SlabPool._free.setdefault(self.device, [])
            fit = [e for e in free if e[0].numel() >= need]
            if fit:
                entry = min(fit, key=lambda e: e[0].numel())
                free[:] = [e for e in free if e is not entry]  # identity, not tensor ==
                chunk, ev = entry
                if ev is not None:
                    torch.cuda.current_stream(self.device).wait_event(ev)
            else:
                chunk = torch.empty(max(need, self.next_floats), dtype=torch.float32, device=self.device)
                self.next_floats = min(self.next_floats * 2, 1 << 30)
            self.chunks.append(chunk)
            self.used = 0
        out = self.chunks[-1][self.used:self.used + nfloats]
        self.used += need
        return out

    def release(self):
        if self.chunks:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(self.device))
            SlabPool._free.setdefault(self.device, []).extend((c, ev) for c in self.chunks)
        self.chunks, self.used = [], 0

    @classmethod
    def trim(cls, device=None):
        """Returns the cached free chunks (of ``device``, or of every device) to the caching allocator."""
        for dev in list(cls._free):
            if device is None or torch.device(device) == dev:
                cls._free[dev] = []


class TableArena:
    """Device memory for kernel argument tables (GEMM problem entries, epilogue tap / group tables), filled
    through a pinned staging mirror with asynchronous copies (a pageable cudaMemcpy per table would synchronise
    the device each time, and must never be captured into a CUDA graph)."""
    ENTRY = ctypes.sizeof(N.GemmProblem)

    def __init__(self, device, capacity=4096):
        self.device, self.nbytes, self.used = torch.device(device), capacity * self.ENTRY, 0
        self.dev = torch.empty(self.nbytes, dtype=torch.uint8, device=self.device)
        self.host = torch.empty(self.nbytes, dtype=torch.uint8).pin_memory()
        self._older = []

    def put(self, raw):
        """Copies ``raw`` (bytes) into the arena (16-byte aligned) and returns the device view."""
        n = len(raw)
        need = (n + 15) // 16 * 16
        if self.used + need > self.nbytes:  # start a fresh block; views into the old one stay valid
            self._older.append((self.dev, self.host))
            self.nbytes = max(self.nbytes, 2 * need)
            self.dev = torch.empty(self.nbytes, dtype=torch.uint8, device=self.device)
            self.host = torch.empty(self.nbytes, dtype=torch.uint8).pin_memory()
            self.used = 0
        lo, hi = self.used, self.used + n
        self.host[lo:hi] = torch.frombuffer(bytearray(raw), dtype=torch.uint8)
        view = self.dev[lo:hi]
        view.copy_(self.host[lo:hi], non_blocking=True)
        self.used += need
        return view


class Planes:
    """hi/lo packed planes of one [rows, K] operand (or several K-concatenated ones)."""

    def __init__(self, rows, k_blocks, device, pool=None):
        self.rows = rows
        self.row_groups = row_groups_of(rows)
        self.k_blocks = k_blocks
        n = self.row_groups * k_blocks * 128
        # no zero-fill needed: pad row groups only feed output rows/cols nobody reads, and the
        # pack kernel writes zeros for k >= K and for rows >= rows inside real groups
        if pool is not None:
            self.hi, self.lo = pool.empty(n), pool.empty(n)
        else:
            self.hi = torch.empty(n, dtype=torch.float32, device=device)
            self.lo = torch.empty(n, dtype=torch.float32, device=device)


def as_rows_view(x, axis):
    """[outer, rows, inner] view of a contiguous tensor for axis `axis` (the reference's
    movedim+reshape, activation_matching.py:26-27, without the copy)."""
    axis = axis % x.dim()
    outer = 1
    for s in x.shape[:axis]:
        outer *= s
    inner = 1
    for s in x.shape[axis + 1:]:
        inner *= s
    return outer, x.shape[axis], inner


def pack_split(x, axis, planes, kb_offset=0, row_index=None, rows=None, sumsq=None, rowsum=None):
    """Packs the [rows, K] operand view of x along `axis` into planes at k-block kb_offset.
    Returns the number of k-blocks written."""
    _require_cuda_f32(x, "pack_split")
    if not x.is_contiguous():
        x = x.contiguous()
    outer, src_rows, inner = as_rows_view(x, axis)
    rows = src_rows if rows is None else rows
    K = outer * inner
    kb = (K + 15) // 16
    if kb_offset + kb > planes.k_blocks or rows > planes.row_groups * 8:
        raise ValueError("pack_split: operand does not fit the planes")
    if PACK_TIMER is not None:  # bench instrumentation: CUDA events around this launch
        e0, e1 = _timer_events()
    N.call("plb_pack_split", x.device, x.data_ptr(), outer, src_rows, inner, N.ptr(row_index), rows,
                                   planes.hi.data_ptr(), planes.lo.data_ptr(), planes.row_groups, kb_offset,
                                   N.ptr(sumsq), N.ptr(rowsum))
    if PACK_TIMER is not None:
        e1.record()
        # algorithmic bytes: every element read once (4 B) and written as a tf32 hi/lo pair (8 B)
        PACK_TIMER.append((e0, e1, 12.0 * rows * outer * inner))
    return kb


def pack_split_pair(xa, xb, axis, pa, pb, sumsq_a=None, sumsq_b=None, sum_a=None, sum_b=None):
    """Packs the two operands of one tap (same shape, all rows) with ONE launch; falls back to two
    ``pack_split`` calls when the geometries differ."""
    _require_cuda_f32(xa, "pack_split_pair")
    _require_cuda_f32(xb, "pack_split_pair")
    if xa.shape != xb.shape or pa.row_groups != pb.row_groups or (sumsq_a is None) != (sumsq_b is None) \
            or (sum_a is None) != (sum_b is None):
        pack_split(xa, axis, pa, sumsq=sumsq_a, rowsum=sum_a)
        pack_split(xb, axis, pb, sumsq=sumsq_b, rowsum=sum_b)
        return
    if not xa.is_contiguous():
        xa = xa.contiguous()
    if not xb.is_contiguous():
        xb = xb.contiguous()
    outer, rows, inner = as_rows_view(xa, axis)
    kb = (outer * inner + 15) // 16
    if kb > min(pa.k_blocks, pb.k_blocks) or rows > pa.row_groups * 8:
        raise ValueError("pack_split_pair: operands do not fit the planes")
    if PACK_TIMER is not None:
        e0, e1 = _timer_events()
    N.call("plb_pack_split_pair_sums", xa.device, xa.data_ptr(), xb.data_ptr(), outer, rows, inner, pa.hi.data_ptr(),
           pa.lo.data_ptr(), pb.hi.data_ptr(), pb.lo.data_ptr(), pa.row_groups, 0, N.ptr(sumsq_a), N.ptr(sumsq_b),
           N.ptr(sum_a), N.ptr(sum_b))
    if PACK_TIMER is not None:
        e1.record()
        PACK_TIMER.append((e0, e1, 2 * 12.0 * rows * outer * inner))


def finalize_grouped_blocks(n):
    """Blocks plb_cross_finalize_grouped uses for an n x n cost matrix: 256-column x 16-row tiles from
    256 units up (1 KB contiguous per partial row), 64-column x 64-row tiles below."""
    cols, rows = (256, 16) if n >= 256 else (64, 64)
    return ((n + cols - 1) // cols) * ((n + rows - 1) // rows)


def choose_bn(n_rows):
    return 64 if n_rows <= 64 else (128 if n_rows <= 128 else 256)


# The tensor core's fp32 accumulator rounds toward zero: measured bias is -1e-7 (relative) per
# 16-wide k-block chained into one accumulator (profiles/experiments/exp_chain_length.py).  A
# chain is therefore capped at MAX_CHAIN_KB k-blocks; the persistent kernel promotes every chain
# into fp32 registers (fully overlapped with the MMAs: chains of 4, 8 or 16 blocks cost the same,
# profiles/r01_notes.md), the v1 kernel cuts K into one CTA per chain and finalize sums in fp64.
MAX_CHAIN_KB = int(os.environ.get("PLB_MAX_CHAIN_KB", "4"))


def choose_splits(tiles, k_blocks, m_rows=128, n_rows=256, impl=None):
    """Number of K splits of one problem.

    Persistent kernel: splits only exist to fill the SMs (small-C taps have a single output tile
    and K up to 401 408); every split costs a partial tile written and re-read, so the count
    minimises a two-term time model (tensor time / wave efficiency + partial traffic).
    v1 kernel: additionally one split per accumulation chain."""
    impl = _GEMM_IMPL if impl is None else impl
    sms = num_sms()
    if impl != "tcgen05":
        fill = min(sms * 4 // max(tiles, 1), k_blocks // 4)
        chain = -(-k_blocks // 16)
        return max(1, min(max(fill, chain), k_blocks))
    max_s = max(1, min(k_blocks // 16, 2 * sms))
    flops = 2.0 * m_rows * n_rows * k_blocks * 16 * tiles
    tile_bytes = 4.0 * m_rows * n_rows * tiles
    best, best_t = 1, None
    for sp in range(1, max_s + 1):
        items = tiles * sp
        eff = items / (-(-items // sms) * sms)
        t = flops / (eff * 120e12) + 2.0 * sp * tile_bytes / 5e12 + 2e-6
        if best_t is None or t < best_t * 0.98:
            best, best_t = sp, t
    return best


class GemmPlan:
    """One 3xTF32 GEMM over packed planes: partial tiles + problem-table entry on device."""

    def __init__(self, a, b, M, Nn, k_blocks, splits=None, symmetric=False, partial=None, pool=None, tables=None):
        self.M, self.N = M, Nn
        self.bn = choose_bn(Nn)
        self.m_tiles = (M + 127) // 128
        self.n_tiles = (Nn + self.bn - 1) // self.bn
        tiles = self.m_tiles * self.n_tiles
        self.symmetric = bool(symmetric)
        active = tiles if not symmetric else sum(
            1 for mt in range(self.m_tiles) for nt in range(self.n_tiles) if 128 * mt + 127 >= self.bn * nt)
        self.splits = choose_splits(active, k_blocks, 128, self.bn) if splits is None else splits
        self.ld_m, self.ld_n = self.m_tiles * 128, self.n_tiles * self.bn
        dev = a.hi.device
        need = self.splits * self.ld_m * self.ld_n
        if partial is None:
            partial = pool.empty(need) if pool is not None else torch.empty(need, dtype=torch.float32, device=dev)
        elif partial.numel() < need:
            raise ValueError("GemmPlan: partial workspace too small")
        self.partial = partial
        self.total_ctas = active * self.splits  # symmetric problems enumerate only their active tiles
        p = N.GemmProblem(a.hi.data_ptr(), a.lo.data_ptr(), b.hi.data_ptr(), b.lo.data_ptr(),
                          self.partial.data_ptr(), a.row_groups, b.row_groups, k_blocks, self.m_tiles,
                          self.n_tiles, self.splits, 0, int(symmetric))
        self.problem = p  # host copy of the table entry (grouped launches re-base cta_begin)
        raw = bytes(p)
        self.table = tables.put(raw) if tables is not None else \
            torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(dev)
        self._keep = (a, b)
        self.alg_flops = 2.0 * M * Nn * k_blocks * 16  # callers that know the unpadded K overwrite

    def run(self, impl=None):
        if GEMM_TIMER is not None:  # bench instrumentation: CUDA events around this launch
            e0, e1 = _timer_events()
            self._launch(impl)
            e1.record()
            GEMM_TIMER.append((e0, e1, self.alg_flops, self.bn, 1))
            return
        self._launch(impl)

    def _launch(self, impl=None):
        N.call("plb_gemm_grouped", self.table.device, self.table.data_ptr(), 1, self.total_ctas, self.bn,
                                         _impl_code(_GEMM_IMPL if impl is None else impl))

    def finalize(self, out, mode=MODE_INNER, qa=None, qb=None, accumulate=False, sa=None, sb=None, K=None):
        """out[i, j] (+)= f(sum_s partial_s[i, j]); out fp32 or fp64 [M, N] (row stride = ldc).  MODE_CORR
        additionally takes the row sums sa / sb and the contraction length K."""
        if mode == MODE_CORR:
            if out.dtype != torch.float32 or sa is None or sb is None or qa is None or qb is None or not K:
                raise ValueError("finalize: the correlation epilogue needs fp32 output, qa/qb, sa/sb and K")
            N.call("plb_cross_finalize_corr", self.partial.device, self.partial.data_ptr(), self.splits, self.ld_m,
                   self.ld_n, self.M, self.N, qa.data_ptr(), qb.data_ptr(), sa.data_ptr(), sb.data_ptr(), int(K),
                   out.data_ptr(), out.stride(0), int(accumulate))
            return
        if out.dtype == torch.float64:
            c32, c64 = None, out.data_ptr()
        else:
            c32, c64 = out.data_ptr(), None
        N.call("plb_cross_finalize", self.partial.device, self.partial.data_ptr(), self.splits, self.ld_m, self.ld_n, self.M,
                                           self.N, N.ptr(qa), N.ptr(qb), mode, c32, c64, out.stride(0),
                                           int(accumulate), self.bn if self.symmetric else 0)


DIRECT_MAX_ROWS = int(os.environ.get("PLB_DIRECT_MAX_ROWS", "128"))  # 0 disables the fused narrow-tap kernel


def direct_gram_eligible(x, y, axis):
    """True when a tap can use the fused narrow-tap kernel (plb_gram_direct): both operands fp32,
    contiguous, 16-byte aligned, the same [outer][C][inner] geometry, C <= 128 a multiple of 8, inner a multiple
    of 16."""
    if DIRECT_MAX_ROWS <= 0 or x.shape != y.shape or x.dtype != torch.float32 or y.dtype != torch.float32:
        return False
    if not (x.is_contiguous() and y.is_contiguous()):
        return False
    if (x.data_ptr() | y.data_ptr()) & 15:  # plb_gram_direct refuses unaligned operands; the packed path takes them
        return False
    outer, rows, inner = as_rows_view(x, axis)
    return rows <= min(DIRECT_MAX_ROWS, 128) and rows % 8 == 0 and inner % 16 == 0 and outer * inner >= 256


class DirectGramPlan:
    """Fused cross-Gram of one narrow tap: partial tiles [splits][128][bn] + the finalize geometry."""

    def __init__(self, rows, K, device, pool=None):
        self.M = self.N = rows
        self.bn = 64 if rows <= 64 else 128
        self.ld_m, self.ld_n = 128, self.bn
        kb = K // 16
        self.splits = max(1, min(num_sms(device), kb // 16))
        need = self.splits * self.ld_m * self.ld_n
        self.partial = pool.empty(need) if pool is not None else torch.empty(need, dtype=torch.float32, device=device)
        self.alg_flops = 2.0 * rows * rows * K
        self.alg_bytes = 2.0 * rows * K * 4
        self.symmetric = False

    def run(self, x, y, axis, qa=None, qb=None):
        outer, rows, inner = as_rows_view(x, axis)
        if DIRECT_TIMER is not None:
            e0, e1 = _timer_events()
        N.call("plb_gram_direct", x.device, x.data_ptr(), y.data_ptr(), outer, rows, inner, self.partial.data_ptr(),
                                        self.splits, MAX_CHAIN_KB, N.ptr(qa), N.ptr(qb))
        if DIRECT_TIMER is not None:
            e1.record()
            DIRECT_TIMER.append((e0, e1, self.alg_bytes, self.alg_flops, rows))

    finalize = GemmPlan.finalize


TMA_GRAM = os.environ.get("PLB_TMA_GRAM", "1") == "1"  # 0: keep the round-1 paths (gram_direct / pack + GEMM)
TMA_MIN_INNER = 16


def tma_gram_eligible(x, y, axis):
    """True when a tap can use the TMA-fed fused kernel (plb_gram_tma): both operands fp32, contiguous,
    16-byte aligned, the same [outer][C][inner] geometry, inner a multiple of 4 (legal tensor-map
    strides) and at least TMA_MIN_INNER (shorter rows waste most of a 32-wide box)."""
    if not TMA_GRAM or x.shape != y.shape or x.dtype != torch.float32 or y.dtype != torch.float32:
        return False
    if not (x.is_cuda and x.is_contiguous() and y.is_contiguous()):
        return False
    if (x.data_ptr() | y.data_ptr()) & 15:
        return False
    outer, rows, inner = as_rows_view(x, axis)
    return rows >= 8 and inner % 4 == 0 and inner >= TMA_MIN_INNER and outer * inner >= 256


def tma_geometry(rows):
    """(cta_group, m_tiles, n_tiles, ld_m, ld_n) of plb_gram_tma for `rows` channels."""
    out = [ctypes.c_int32() for _ in range(5)]
    rc = N.lib().plb_gram_tma_geometry(rows, *[ctypes.byref(v) for v in out])
    if rc != 0:
        raise RuntimeError("plb_gram_tma_geometry failed")
    return tuple(v.value for v in out)


def choose_tma_splits(tiles, cta_group, total_boxes, tile_elems, sms):
    """K splits of a TMA-fed Gram: fill the SM clusters; every split costs one partial tile written
    and re-read by the epilogue, every work item a pipeline ramp."""
    clusters = max(1, sms // cta_group)
    max_s = max(1, min(total_boxes // 4, 4 * clusters))
    best, best_t = 1, None
    mma_s_per_box = 12 * 128 / 1.9e9  # 12 tcgen05.mma of 128 clocks per 32-wide box
    for sp in range(1, max_s + 1):
        items = tiles * sp
        rounds = -(-items // clusters)
        boxes = -(-total_boxes // sp)
        t = rounds * (boxes * mma_s_per_box + 4e-6) + 2.0 * sp * tiles * tile_elems * 4 / 4e12
        if best_t is None or t < best_t * 0.98:
            best, best_t = sp, t
    return best


# Longest contraction one work item of plb_gram_tma walks, whatever split count the fill model or the caller asks
# for.  An item accumulates in fp32 before its sums reach fp64 (the Gram in the promotion registers once per chain,
# the row moments per converter lane, 4 values per box), and a long fp32 sum stagnates: measured on a B200 with
# post-ReLU data, one item over K = 2^25 is off by 5e-5 in the Gram and 1.5e-3 in the sums of squares, and an item of
# 14 364 boxes (what the fill model picks for C = 256, K = 2^25) by 2.6e-6 in the sums of squares; items of up to
# 890 boxes stay below 7e-7 and 1e-7.  Taps of a batch of 32 walk at most ~90 boxes per item, so the cap never binds
# there.
TMA_MAX_K_PER_ITEM = 512 * 32


class TmaGramPlan:
    """TMA-fed fused cross-Gram of one tap (any width): partial tiles + the finalize geometry.  ``splits`` (default:
    ``choose_tma_splits``) is raised where needed so that no work item walks more than TMA_MAX_K_PER_ITEM of K."""

    def __init__(self, rows, outer, inner, device, pool=None, splits=None):
        self.M = self.N = rows
        self.cta_group, self.m_tiles, self.n_tiles, self.ld_m, self.ld_n = tma_geometry(rows)
        self.bn = self.ld_n // self.n_tiles
        K = outer * inner
        total_boxes = outer * ((inner + 31) // 32)
        tiles = self.m_tiles * self.n_tiles
        tile_elems = (self.ld_m // self.m_tiles) * self.bn
        self.splits = splits if splits is not None else \
            choose_tma_splits(tiles, self.cta_group, total_boxes, tile_elems, num_sms(device))
        self.splits = max(self.splits, -(-total_boxes * 32 // TMA_MAX_K_PER_ITEM))
        need = self.splits * self.ld_m * self.ld_n
        self.partial = pool.empty(need) if pool is not None else torch.empty(need, dtype=torch.float32, device=device)
        self.alg_flops = 2.0 * rows * rows * K
        self.alg_bytes = 2.0 * rows * K * 4
        self.symmetric = False

    def run(self, x, y, axis, qa=None, qb=None, sa=None, sb=None):
        outer, rows, inner = as_rows_view(x, axis)
        if DIRECT_TIMER is not None:
            e0, e1 = _timer_events()
        N.call("plb_gram_tma", x.device, x.data_ptr(), y.data_ptr(), outer, rows, inner, self.partial.data_ptr(),
               self.splits, MAX_CHAIN_KB, N.ptr(qa), N.ptr(qb), N.ptr(sa), N.ptr(sb))
        if DIRECT_TIMER is not None:
            e1.record()
            DIRECT_TIMER.append((e0, e1, self.alg_bytes, self.alg_flops, rows))

    finalize = GemmPlan.finalize


class GroupedGemm:
    """Several small problems of one tile width in ONE persistent launch (their CTAs share the
    148 SMs), e.g. the ~100 small taps of a ResNet-50 calibration batch."""

    def __init__(self, plans, tables=None):
        assert plans and len({p.bn for p in plans}) == 1
        self.plans, self.bn = list(plans), plans[0].bn
        raw, begin = bytearray(), 0
        for p in self.plans:
            q = N.GemmProblem.from_buffer_copy(bytes(p.problem))
            q.cta_begin = begin
            begin += p.total_ctas
            raw += bytes(q)
        self.total_items = begin
        self.table = tables.put(bytes(raw)) if tables is not None else \
            torch.frombuffer(raw, dtype=torch.uint8).to(self.plans[0].partial.device)
        self.alg_flops = sum(p.alg_flops for p in self.plans)

    def run(self, impl=None):
        name = _GEMM_IMPL if impl is None else impl
        if GEMM_TIMER is not None:
            e0, e1 = _timer_events()
        N.call("plb_gemm_grouped", self.table.device, self.table.data_ptr(), len(self.plans), self.total_items, self.bn,
                                         _impl_code(name))
        if GEMM_TIMER is not None:
            e1.record()
            GEMM_TIMER.append((e0, e1, self.alg_flops, self.bn, len(self.plans)))


def cross_statistic(x, y, axis, mode):
    """One tap: [x.shape[axis], y.shape[axis]] cross-statistic matrix of two activations
    (cross_features_inner_product / cross_features_cdist, activation_matching.py:14-46; MODE_CORR: the
    Pearson correlation of the unit pairs)."""
    _require_cuda_f32(x, "cross_statistic")
    _require_cuda_f32(y, "cross_statistic")
    oa, ra, ia = as_rows_view(x, axis)
    ob, rb, ib = as_rows_view(y, axis)
    if oa * ia != ob * ib:
        raise ValueError(f"cross_statistic: contraction sizes differ ({oa * ia} vs {ob * ib})")
    K = oa * ia
    kb = (K + 15) // 16
    dev = x.device
    qa = qb = sa = sb = None
    if mode != MODE_INNER:  # fp64 row moments: [qa | qb | sa | sb]
        q = torch.zeros(2 * (ra + rb), dtype=torch.float64, device=dev)
        qa, qb = q[:ra], q[ra:ra + rb]
        if mode == MODE_CORR:
            sa, sb = q[ra + rb:2 * ra + rb], q[2 * ra + rb:]
    out = torch.empty(ra, rb, dtype=torch.float32, device=dev)
    if tma_gram_eligible(x, y, axis):  # TMA-fed fused kernel straight from the activations, no packed planes
        plan = TmaGramPlan(ra, oa, ia, dev)
        plan.run(x, y, axis, qa, qb, sa, sb)
        plan.finalize(out, mode, qa, qb, accumulate=False, sa=sa, sb=sb, K=K)
        return out
    if mode != MODE_CORR and direct_gram_eligible(x, y, axis):  # round-1 narrow-tap kernel (PLB_TMA_GRAM=0)
        plan = DirectGramPlan(ra, K, dev)
        plan.run(x, y, axis, qa, qb)
        plan.finalize(out, mode, qa, qb, accumulate=False)
        return out
    pa, pb = Planes(ra, kb, dev), Planes(rb, kb, dev)
    pack_split_pair(x, y, axis, pa, pb, qa, qb, sa, sb)
    plan = GemmPlan(pa, pb, ra, rb, kb)
    plan.run()
    plan.finalize(out, mode, qa, qb, accumulate=False, sa=sa, sb=sb, K=K)
    return out


# ------------------------------------------------------------------------------------ LAP

LAP_MAX_N = 4096  # plb_lap_solve_batched / plb_get_blocks keep all per-unit state in shared memory


def lap_solve_batched(costs, maximize=True, v_init=None, v_scale=1.0, return_duals=False):
    """Solves all square problems in one launch.  Returns (list of int64 CUDA tensors,
    objective fp64 CUDA tensor, status int32 CUDA tensor[, list of fp64 column-dual tensors]).

    ``v_init`` (list with one fp64 CUDA tensor [n] or None per problem) warm-starts the solver from the column
    duals of a related problem (``return_duals=True`` of an earlier call), scaled by ``v_scale``: same optimum, far
    fewer augmenting steps when the problem changed little; SciPy's tie-breaking is only reproduced cold."""
    if not costs:
        return ([], None, None, []) if return_duals else ([], None, None)
    dev = costs[0].device
    mats = []
    for c in costs:
        _require_cuda_f32(c, "lap_solve_batched")
        if c.dim() != 2 or c.shape[0] != c.shape[1]:
            raise ValueError(f"lap_solve_batched: square cost matrices only, got {tuple(c.shape)}")
        mats.append(c if c.stride(1) == 1 else c.contiguous())
    ns = [m.shape[0] for m in mats]
    if max(ns) > LAP_MAX_N:
        raise ValueError(f"lap_solve_batched: a permutation group has {max(ns)} units; the shared-memory assignment "
                         f"kernel holds at most {LAP_MAX_N} (45 B of solver state per unit in 227 KB)")
    outs = [torch.empty(n, dtype=torch.int64, device=dev) for n in ns]
    warm = v_init is not None or return_duals
    rows = [[m.data_ptr() for m in mats], [o.data_ptr() for o in outs]]
    duals = None
    if warm:
        vin = list(v_init) if v_init is not None else [None] * len(mats)
        for v, n in zip(vin, ns):
            if v is not None and not (v.is_cuda and v.dtype == torch.float64 and v.numel() == n and v.is_contiguous()):
                raise ValueError("lap_solve_batched: v_init entries must be contiguous fp64 CUDA tensors of length n")
        duals = [torch.empty(n, dtype=torch.float64, device=dev) for n in ns] if return_duals else None
        rows.append([0 if v is None else v.data_ptr() for v in vin])
        rows.append([d.data_ptr() for d in duals] if duals is not None else [0] * len(mats))
    table = torch.tensor(rows, dtype=torch.int64).to(dev)
    meta = torch.tensor([ns, [m.stride(0) for m in mats]], dtype=torch.int32).to(dev)
    obj = torch.empty(len(mats), dtype=torch.float64, device=dev)
    status = torch.empty(len(mats), dtype=torch.int32, device=dev)
    if warm:
        N.call("plb_lap_solve_batched_warm", dev, table[0].data_ptr(), meta[0].data_ptr(), meta[1].data_ptr(),
               table[1].data_ptr(), obj.data_ptr(), status.data_ptr(), len(mats), max(ns), int(bool(maximize)),
               table[2].data_ptr(), float(v_scale), table[3].data_ptr() if duals is not None else None)
        if return_duals:
            return outs, obj, status, duals
        return outs, obj, status
    N.call("plb_lap_solve_batched", dev, table[0].data_ptr(), meta[0].data_ptr(), meta[1].data_ptr(),
           table[1].data_ptr(), obj.data_ptr(), status.data_ptr(), len(mats), max(ns), int(bool(maximize)))
    return outs, obj, status


def raise_on_lap_status(status):
    st = status.cpu()
    if (st == 2).any():
        raise ValueError("matrix contains invalid numeric entries")  # SciPy's message
    if (st == 1).any():
        raise ValueError("cost matrix is infeasible")


# ------------------------------------------------------------------------------------ blocks

def get_blocks_launch(cost, perm, ratio, identity, buf, count):
    """Enqueues get_blocks for one group (partial_matching.py:76-86) into caller-provided buffers: buf int64
    [4, n] receives Q[mask], P[mask], Q[~mask], P[~mask] (order-preserving, front-packed), count int32[1] the
    number of merged units.  No synchronisation."""
    _require_cuda_f32(cost, "get_blocks")
    n = cost.shape[0]
    N.call("plb_get_blocks", cost.device, cost.data_ptr(), cost.stride(0), perm.data_ptr(), n, float(ratio),
           int(identity), buf[0].data_ptr(), buf[1].data_ptr(), buf[2].data_ptr(), buf[3].data_ptr(), count.data_ptr())


def get_blocks_group(cost, perm, ratio, identity):
    """(Q[mask], P[mask], Q[~mask], P[~mask]) for one group (partial_matching.py:76-86)."""
    n = cost.shape[0]
    dev = cost.device
    buf = torch.empty(4, n, dtype=torch.int64, device=dev)
    counts = torch.zeros(1, dtype=torch.int32, device=dev)
    perm = perm.to(device=dev, dtype=torch.int64).contiguous()
    get_blocks_launch(cost, perm, ratio, identity, buf, counts)
    m = int(counts.item())
    return buf[0, :m], buf[1, :m], buf[2, :n - m], buf[3, :n - m]


def _prod(xs):
    r = 1
    for v in xs:
        r *= v
    return r


def block_merge(w1, w2, blocks_by_axis):
    """Assembles one merged tensor (partial_matching.py:112-176).  blocks_by_axis maps the
    tensor's blocked axes ({0}, {1}, {k} or {0, 1}) to (b1, b2, b1c, b2c) int64 CUDA index
    tensors."""
    _require_cuda_f32(w1, "block_merge")
    _require_cuda_f32(w2, "block_merge")
    w1, w2 = w1.contiguous(), w2.contiguous()
    shape = list(w1.shape)
    axes = sorted(blocks_by_axis)
    if axes == [0, 1]:
        bo, bi, in_only = blocks_by_axis[0], blocks_by_axis[1], 0
        O, I, R = shape[0], shape[1], _prod(shape[2:])
    elif axes == [0]:
        bo, bi, in_only = blocks_by_axis[0], None, 0
        O, I, R = shape[0], 1, _prod(shape[1:])
    elif len(axes) == 1:  # concatenation along a non-leading axis (partial_matching.py:122-129)
        ax = axes[0]
        bo, bi, in_only = None, blocks_by_axis[ax], 1
        O, I, R = _prod(shape[:ax]), shape[ax], _prod(shape[ax + 1:])
    else:
        raise ValueError(f"block_merge: unsupported blocked axes {axes}")

    keep = []

    def unpack(b):
        if b is None:
            return [None, None, None, None], 0, 0
        b = [t.to(device=w1.device, dtype=torch.int64).contiguous() for t in b]
        keep.append(b)
        return [t.data_ptr() if t.numel() else None for t in b], b[0].numel(), b[2].numel()

    po, no, mo = unpack(bo)
    pi, ni, mi = unpack(bi)
    if bo is not None and no == 0 or bi is not None and ni == 0:
        raise ValueError("block_merge: a blocked axis needs at least one merged unit")
    Oout = no + 2 * mo if bo is not None else O
    Iout = ni + 2 * mi if bi is not None else I
    out = torch.empty(Oout * Iout * R, dtype=torch.float32, device=w1.device)
    N.call("plb_block_merge", w1.device, w1.data_ptr(), w2.data_ptr(), O, I, R, po[0], po[1], po[2], po[3], no, mo,
                                    pi[0], pi[1], pi[2], pi[3], ni, mi, in_only, out.data_ptr())
    if axes == [0, 1]:
        return out.view([Oout, Iout] + shape[2:])
    if axes == [0]:
        return out.view([Oout] + shape[1:])
    return out.view(shape[:axes[0]] + [Iout] + shape[axes[0] + 1:])


def gather_axis(x, axis, P):
    """index_select(x, axis, P) (apply_perm, pleas/core/utils.py:244)."""
    _require_cuda_f32(x, "gather_axis")
    x = x.contiguous()
    outer, n, inner = as_rows_view(x, axis)
    P = P.to(device=x.device, dtype=torch.int64).contiguous()
    out_shape = list(x.shape)
    out_shape[axis % x.dim()] = P.numel()
    if P.numel() != n:
        raise ValueError("gather_axis: permutation length mismatch")
    out = torch.empty(out_shape, dtype=torch.float32, device=x.device)
    N.call("plb_gather_axis", x.device, x.data_ptr(), out.data_ptr(), outer, n, inner, P.data_ptr())
    return out


def compose_perm(a, b):
    out = torch.empty_like(a)
    N.call("plb_compose_perm", a.device, a.data_ptr(), b.data_ptr(), out.data_ptr(), a.numel())
    return out


def wm_progress(A, P, flag, gain=None):
    N.call("plb_wm_progress", A.device, A.data_ptr(), A.stride(0), P.data_ptr(), A.shape[0], flag.data_ptr(),
                                    N.ptr(gain))


# ------------------------------------------------------------------------------------ solve

def chol_solve_(G, B, ridge):
    """In place: G <- chol(G + ridge I) (lower), B <- (G + ridge I)^-1 B.  fp64 CUDA, row-major."""
    assert G.dtype == torch.float64 and B.dtype == torch.float64 and G.is_cuda and B.is_cuda
    assert G.is_contiguous() and B.is_contiguous() and G.shape[0] == G.shape[1] == B.shape[0]
    info = torch.zeros(1, dtype=torch.int32, device=G.device)
    N.call("plb_chol_solve", G.device, G.data_ptr(), G.shape[0], B.data_ptr(), B.shape[1], float(ridge),
                                   info.data_ptr())
    return info


# ------------------------------------------------------------------------------------ im2col

def pack_im2col(x1, x2, chan1, chan2, scale1, scale2, cmerged, kernel, stride, padding, dilation, out_hw,
                ones_row, planes, kb_offset=0):
    """Packs rows f=(c,dy,dx) x k=(n,ho,wo) of the merged layer input
    s1[c]*x1[:, chan1[c]] + s2[c]*x2[:, chan2[c]] (pleas_merging.py:116-123, 146-147) into planes.
    x1/x2: [N, C, H, W] float32 CUDA (x2 may be None)."""
    _require_cuda_f32(x1, "pack_im2col")
    x1 = x1.contiguous()
    if x2 is not None:
        _require_cuda_f32(x2, "pack_im2col")
        x2 = x2.contiguous()
        assert x2.shape == x1.shape
    Nb, C, H, W = x1.shape
    Ho, Wo = out_hw
    N.call("plb_pack_im2col", x1.device, x1.data_ptr(), N.ptr(x2), Nb, C, H, W, N.ptr(chan1), N.ptr(chan2),
                                    N.ptr(scale1), N.ptr(scale2), cmerged, kernel[0], kernel[1], stride[0],
                                    stride[1], padding[0], padding[1], dilation[0], dilation[1], Ho, Wo,
                                    int(bool(ones_row)), planes.hi.data_ptr(), planes.lo.data_ptr(),
                                    planes.row_groups, kb_offset)
