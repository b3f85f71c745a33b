// Forward convolution of the source models as a 3xTF32 implicit GEMM on tcgen05 (include/pleas_b200.h,
// plb_conv2d_forward).  Replaces the ATen / cuDNN fp32 convolutions the reference's loops run
// (pleas/methods/activation_matching.py:123, pleas_merging.py:262-281) — SIMT kernels at ~38 TFLOP/s that
// were 60 % of a calibration step.
//
// GEMM view (NCHW fp32, no layout change anywhere):
//     D[p, co] = sum_k A[p, k] B[co, k]      p = (n, oh, ow) output position      -> M (tile 128 = TMEM lanes)
//                                            co output channel                    -> N (tile TN = 64 / 128)
//                                            k = (32-channel block, kh, kw)       -> K in boxes of 32
// Positions are the M dimension because they are the contiguous dimension of both x and out: a warp's
// loads (32 consecutive positions of one channel) and stores (32 consecutive positions of one output
// channel) are 128-byte coalesced with no transposition.
//
//   A (activations): loader threads own one position each.  They gather their 32 channels of the current
//     tap with 4-byte cp.async (zero padding = zero-size copies) into a private shared-memory ring that is
//     several stages deep — the prefetch needs no registers and no cross-thread synchronisation, every
//     thread reads back only what it copied — then split in registers (hi = rna_tf32(x),
//     lo = rna_tf32(x - hi)) and write both planes into TENSOR MEMORY with tcgen05.st: the MMA takes A from
//     TMEM (tcgen05.mma [d], [a], b_desc).  That is the operand arrangement the shared-memory-bound Gram
//     kernel's analysis asked for (profiles/r02_notes.md): the MMAs read only the B operand from shared
//     memory, the raw A stream crosses it once.
//   B (weights) is packed ONCE per model (plb_conv_pack_weights: hi / lo planes, [tap][Cout][Cin]) and
//     arrives by 4-D tensor-map TMA in the 128-byte-swizzled K-major layout.
//   D: the tensor core's fp32 accumulator truncates, so K is cut into short chains; the MMA warp ping-pongs
//     between two TMEM accumulators and the epilogue warps promote every finished chain into registers
//     (same scheme as gemm.cu / gram_tma.cu), then store the tile (+ bias) straight into NCHW.
//
// TMEM columns: [0, 2 TN) accumulators, [2 TN, 2 TN + 4 x 64) four A stages (hi | lo, 32 k each).
// Warp roles (576 threads, 1 CTA/SM, persistent over (position tile, model, channel tile) items):
//   warp 0       TMA producer (weights)          warp 1        TMEM owner + MMA issuer
//   warps 2-9    loaders: two per TMEM lane quadrant, 16 of a box's 32 channels each (a single warp per
//                quadrant was the critical path: ~630 instructions per stage, profiles/r02_notes.md)
//   warps 10-17  promotion / epilogue (two per lane quadrant, half the channel tile each)
#include "tma.cuh"

namespace plb {

constexpr int kConvStages = 4;
constexpr int kConvThreads = 576;
constexpr int kConvMaxFlatK = 512;  // flat form: K = Cin*KH*pow2(KW) padded to 32; bounds the kernel-row table (KW <= 16)

struct ConvParams {
  const float *x[2];
  const float *bias[2];
  float *out[2];
  const float2 *post[2];  // per output channel (scale, shift) of the fused per-channel affine, or nullptr
  float *out2[2];         // second output: relu?(scale * out + shift)
  int post_relu;
  int nprob;
  int NB, Cin, IH, IW, Cout, OH, OW, KH, KW, stride, pad_h, pad_w;
  int P, OHW, IHW;
  int m_tiles, n_tiles, total_items;
  int taps;         // KH*KW (channel-block form) or 1 (flat form)
  int nbox;         // K boxes of 32 per item
  int flat;         // 1: k = (ci*KH + kh) * KWP + kw (any Cin; KWP = KW rounded up to a power of two), 0: k = 32-channel block x tap
  int flat_groups;  // Cin*KH kernel rows (flat form)
  int flat_lg;      // log2(KWP)
  int chain_boxes;  // boxes chained into one TMEM accumulator before promotion
  unsigned long long *trace;  // experiments only (plb_conv_debug_set_trace): 8 clock64 stamps per box of CTA 0
  int debug;        // experiments only (PLB_CONV_DEBUG, WRONG results): 1 no gather, 2 one MMA of three, 4 no stores
};

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}
// D[tmem] (+)= A[tmem] * B[smem desc], kind::tf32 (A: lane = row, column = k)
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void *smem_dst, const CUtensorMap *map, int c0, int c1, int c2, int c3,
                                            uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], "
      "[%6];" ::"r"(smem_u32(smem_dst)),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(smem_u32(bar))
      : "memory");
}

template <int TN>
struct ConvCfg {
  static constexpr int kBBytes = kConvStages * 2 * TN * 128;
  static constexpr int kARing = TN == 128 ? 5 : 8;
  static constexpr int kSmemBytes = kBBytes + kARing * 16384 + 1024;
};

// 4-byte cp.async; `ignore` != 0 writes zeros instead of reading src (the convolution's zero padding)
__device__ __forceinline__ void cp_async4(uint32_t smem_dst, const float *src, uint32_t ignore) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %2, 0;\n\t"
      "cp.async.ca.shared.global [%0], [%1], 4, p;\n\t}" ::"r"(smem_dst),
      "l"(src), "r"(ignore)
      : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// Barrier helpers on raw 32-bit shared addresses.  The kernel computes ONE opaque base (asm volatile, so the
// compiler keeps it in a register) for all its barriers: re-deriving `&bar[s]` costs an S2R SR_CgaCtaId plus
// address arithmetic at every use, and on the MMA-issuing warp every clock between two boxes is an idle
// tensor core (profiles/r02_notes.md).
__device__ __forceinline__ uint32_t opaque_smem_u32(const void *p) {
  uint32_t a;
  asm volatile("{\n\t.reg .u64 t;\n\tcvta.to.shared.u64 t, %1;\n\tcvt.u32.u64 %0, t;\n\t}" : "=r"(a) : "l"(p));
  return a;
}
__device__ __forceinline__ void a32_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void a32_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool a32_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// non-blocking probe (try_wait may suspend the thread for a while when the phase is still open)
__device__ __forceinline__ bool a32_test_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void a32_wait_wd(uint32_t bar, uint32_t parity) {
  if (a32_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!a32_try_wait(bar, parity))
    if (clock64() - t0 > kWatchdogClocks) __trap();
}
__device__ __forceinline__ void a32_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void a32_tma_load_4d(uint32_t smem_dst, const CUtensorMap *map, int c0, int c1, int c2,
                                                int c3, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], "
      "[%6];" ::"r"(smem_dst),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar)
      : "memory");
}

// flat-form gather of one loader thread: 16 >> LG kernel rows of (1 << LG) taps (see conv3xtf32_kernel)
template <int LG>
__device__ __forceinline__ void flat_rows(const int2 *rows, const float *origin, const float *safe, uint32_t dst,
                                          bool pvalid, int ih0, int iw0, int IH, int IW, int KW) {
  constexpr int TAPS = 1 << LG, ROWS = 16 >> LG;
#pragma unroll
  for (int r = 0; r < ROWS; ++r) {
    const int2 e = rows[r];
    const bool rowok = pvalid && e.y >= 0 && (unsigned)(ih0 + e.y) < (unsigned)IH;
    const float *base = rowok ? origin + e.x : safe;
#pragma unroll
    for (int t = 0; t < TAPS; ++t) {
      const bool ok = rowok && t < KW && (unsigned)(iw0 + t) < (unsigned)IW;
      cp_async4(dst + (r * TAPS + t) * 512, base + (ok ? t : 0), ok ? 0u : 1u);
    }
  }
}

// epilogue stores of one thread: its position's COLS channel values (stride ohw between channels)
template <int COLS, bool BIAS, bool POST>
__device__ __forceinline__ void store_tile(const float (&acc)[COLS], float *o, float *o2, int ohw, const float *bias,
                                           const float2 *ss, bool relu, int) {
#pragma unroll
  for (int c = 0; c < COLS; ++c) {
    const float v = acc[c];
    o[(int64_t)c * ohw] = v;
    if (POST) {
      const float2 a = __ldg(ss + c);
      const float w = fmaf(v, a.x, a.y);
      o2[(int64_t)c * ohw] = relu ? fmaxf(w, 0.f) : w;
    }
  }
}
template <int COLS>
__device__ __noinline__ void store_tile_ragged(const float (&acc)[COLS], float *o, float *o2, int ohw, const float *bias,
                                               const float2 *ss, bool relu, int nc) {
#pragma unroll 4
  for (int c = 0; c < COLS; ++c) {
    if (c >= nc) break;
    const float v = acc[c] + (bias ? __ldg(bias + c) : 0.f);
    o[(int64_t)c * ohw] = v;
    if (o2 != nullptr) {
      const float2 a = __ldg(ss + c);
      const float w = fmaf(v, a.x, a.y);
      o2[(int64_t)c * ohw] = relu ? fmaxf(w, 0.f) : w;
    }
  }
}

struct ConvItem {
  int prob, mt, nt;
};
__device__ __forceinline__ ConvItem conv_item(const ConvParams &p, int item) {
  ConvItem it;
  it.nt = item % p.n_tiles;
  const int rest = item / p.n_tiles;
  it.prob = rest % p.nprob;
  it.mt = rest / p.nprob;
  return it;
}

// TN: output-channel tile; CH: boxes per accumulation chain; DBG: experiments build (trace stamps, PLB_CONV_DEBUG)
template <int TN, int CH, bool DBG>
__global__ void __launch_bounds__(kConvThreads, 1) conv3xtf32_kernel(const __grid_constant__ CUtensorMap tmw0,
                                                                      const __grid_constant__ CUtensorMap tmw1,
                                                                      ConvParams p) {
  constexpr int kPlaneBytes = TN * 128;          // one (TN rows x 32 k) weight box
  constexpr int kStageBytes = 2 * kPlaneBytes;   // hi | lo
  constexpr uint32_t kACol0 = 2 * TN;            // first TMEM column of the A stages
  constexpr int kARing = ConvCfg<TN>::kARing;    // depth of the loaders' cp.async ring ([c][row] fp32, 16 KB / stage)
  extern __shared__ uint8_t smem_raw[];
  // [0,4) full: TMA (weights, tx bytes) + the eight loader warps (A in TMEM) -> MMA;  [4,8) empty: MMA -> producer
  // and loaders;  [8,10) accumulator full: MMA -> promotion warps;  [10,12) accumulator empty: promotion -> MMA
  __shared__ uint64_t bars[2 * kConvStages + 4];
  __shared__ uint32_t tmem_base_s;
  __shared__ int2 ktab[kConvMaxFlatK];           // flat form: kernel row g = ci*KH + kh -> (ci*IHW + kh*IW, kh) or (0, -1)

  uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cta = (int)blockIdx.x, nctas = (int)gridDim.x;
  const uint32_t bars_a = opaque_smem_u32(bars), smem_a = opaque_smem_u32(smem);
  const uint32_t bar_full = bars_a, bar_empty = bars_a + 8 * kConvStages, bar_acc_full = bars_a + 16 * kConvStages,
                 bar_acc_empty = bar_acc_full + 16;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < kConvStages; ++s) {
      mbar_init(&bars[s], 1 + 8);
      mbar_init(&bars[kConvStages + s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&bars[2 * kConvStages + b], 1);
      mbar_init(&bars[2 * kConvStages + 2 + b], 8);
    }
    fence_mbar_init();
  } else if (warp == 1) {
    tmem_alloc(&tmem_base_s, 512);
    tmem_relinquish();
  }
  if (p.flat) {
    const int rows = (p.nbox * 32) >> p.flat_lg;  // kernel rows incl. the zero rows that pad K to a box multiple
    for (int g = (int)threadIdx.x; g < rows; g += kConvThreads) {
      int2 e;
      if (g < p.flat_groups) {
        const int ci = g / p.KH, kh = g - ci * p.KH;
        e.x = ci * p.IHW + kh * p.IW;
        e.y = kh;
      } else {
        e.x = 0;
        e.y = -1;  // padding rows always read as zero
      }
      ktab[g] = e;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (weights)
    uint32_t i = 0;
    for (int item = cta; item < p.total_items; item += nctas) {
      const ConvItem it = conv_item(p, item);
      const CUtensorMap *map = it.prob ? &tmw1 : &tmw0;
      const int n0 = it.nt * TN;
      int cb = 0, tap = 0;
      for (int b = 0; b < p.nbox; ++b, ++i) {
        const uint32_t s = i & (kConvStages - 1), ph = (i / kConvStages) & 1u;
        a32_wait_wd(bar_empty + 8 * s, ph ^ 1u);
        if (DBG && p.trace && cta == 0 && lane == 0 && i < 512) p.trace[i * 16 + 0] = clock64();
        if (elect_one()) {
          const uint32_t st = smem_a + s * kStageBytes;
          a32_expect_tx(bar_full + 8 * s, kStageBytes);
          a32_tma_load_4d(st, map, cb * 32, n0, tap, 0, bar_full + 8 * s);
          a32_tma_load_4d(st + kPlaneBytes, map, cb * 32, n0, tap, 1, bar_full + 8 * s);
        }
        __syncwarp();
        if (++tap == p.taps) {
          tap = 0;
          ++cb;
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc = umma_idesc_tf32(128, TN);
    const uint32_t smem_base = smem_a;
    // Every clock this warp spends between the last MMA of a chain and the first of the next is an idle tensor
    // core, and the SM's issue slots are contended by sixteen busy loader / promotion warps (a barrier probe
    // costs 100-250 clocks here, profiles/r02_notes.md).  So: one barrier per stage for A and B, the next
    // chain's barriers are probed (non-blocking test_wait) BEFORE this chain's MMAs are issued, and barrier
    // addresses are plain registers.
    // A chain = up to chain_boxes consecutive boxes into one accumulator.  All small products of the chain are
    // issued first: while the accumulator only holds lo x hi terms (2^-11 of the final magnitude) the tensor
    // core's truncating adds cost nothing, so only the hi x hi MMAs add at full magnitude.
    uint32_t i = 0, chain = 0;
    uint32_t ready = 0;   // bit q: box i + q's barrier was already seen complete
    bool acc_ok = false;  // the next chain's accumulator was already seen drained
    for (int item = cta; item < p.total_items; item += nctas) {
      for (int b0 = 0; b0 < p.nbox; b0 += CH, ++chain) {
        const uint32_t buf = chain & 1u;
        const int nb = min(CH, p.nbox - b0);
        const bool trm = DBG && p.trace && cta == 0 && lane == 0 && i < 512;
        if (trm) p.trace[i * 16 + 8] = clock64();
        if (!acc_ok) a32_wait_wd(bar_acc_empty + 8 * buf, ((chain >> 1) & 1u) ^ 1u);
        const uint32_t d_tmem = tmem_base + buf * TN;
#pragma unroll
        for (int q = 0; q < CH; ++q)
          if (q < nb && !((ready >> q) & 1u)) a32_wait_wd(bar_full + 8 * ((i + q) & (kConvStages - 1)), ((i + q) / kConvStages) & 1u);
        if (trm) p.trace[i * 16 + 4] = clock64();
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int q = 0; q < CH; ++q) {
            if (q >= nb) break;
            const uint32_t s = (i + q) & (kConvStages - 1);
            const uint32_t bst = smem_base + s * kStageBytes, a_hi0 = tmem_base + kACol0 + s * 64;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              umma_tf32_ts(d_tmem, a_hi0 + 32 + 8 * j, umma_desc_sw<128>(bst + 32 * j), idesc, (q > 0 || j > 0) ? 1u : 0u);
              if (!(DBG && p.debug & 2))
                umma_tf32_ts(d_tmem, a_hi0 + 8 * j, umma_desc_sw<128>(bst + kPlaneBytes + 32 * j), idesc, 1u);
            }
          }
        }
        __syncwarp();
        // Probes for the next chain, issued BETWEEN the chain's two MMA phases: the stages of the next chain are
        // the ones the previous chain released when this one started executing, so at the top of the chain the
        // loaders have not refilled them yet (the probe would always fail and the blocking wait after the issue
        // loop would cost 100-250 clocks per barrier); two thirds of the chain's MMAs later they have, and the
        // tensor pipe keeps draining its queue while the probes are in flight.  Harmless when there is no next
        // chain: they just report "not yet".
        uint32_t nready = 0;
#pragma unroll
        for (int q = 0; q < CH; ++q) {
          const uint32_t in = i + nb + q;
          if (a32_test_wait(bar_full + 8 * (in & (kConvStages - 1)), (in / kConvStages) & 1u)) nready |= 1u << q;
        }
        const bool next_acc = a32_test_wait(bar_acc_empty + 8 * ((chain + 1) & 1u), (((chain + 1) >> 1) & 1u) ^ 1u);
        if (elect_one()) {
#pragma unroll
          for (int q = 0; q < CH; ++q) {
            if (q >= nb) break;
            const uint32_t s = (i + q) & (kConvStages - 1);
            const uint32_t bst = smem_base + s * kStageBytes, a_hi0 = tmem_base + kACol0 + s * 64;
            if (!(DBG && p.debug & 2)) {
#pragma unroll
              for (int j = 0; j < 4; ++j) umma_tf32_ts(d_tmem, a_hi0 + 8 * j, umma_desc_sw<128>(bst + 32 * j), idesc, 1u);
            }
            a32_commit(bar_empty + 8 * s);
          }
          a32_commit(bar_acc_full + 8 * buf);
        }
        ready = __reduce_and_sync(0xffffffffu, nready);
        acc_ok = __all_sync(0xffffffffu, next_acc);
        if (trm) p.trace[i * 16 + 6] = clock64();
        i += nb;
      }
    }
  } else if (warp < 10) {
    // ------------------------------------------------------------------ loaders (A operand -> TMEM)
    const int hsel = (warp - 2) >> 2;        // which 16 channels of every 32-channel box
    const int row = (warp & 3) * 32 + lane;  // TMEM lane = position inside the tile
    const uint32_t a_base = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + kACol0 + 16 * hsel;
    // ring slot layout [c][row] fp32: + slot * 16 KB + c * 512
    const uint32_t ring = smem_a + ConvCfg<TN>::kBBytes + (uint32_t)(hsel * 16) * 512u + (uint32_t)row * 4u;
    const int my_items = cta < p.total_items ? (p.total_items - cta + nctas - 1) / nctas : 0;
    const int total = my_items * p.nbox;
    // issue-side cursor: work item, channel block, tap
    const int kh_n = p.flat ? 1 : p.KH, kw_n = p.flat ? 1 : p.KW, cb_n = p.nbox / (kh_n * kw_n);
    int itx = 0, cb = 0, kh = 0, kw = 0, ih0 = 0, iw0 = 0;
    bool pvalid = false;
    const float *xn = nullptr;
    auto locate = [&]() {  // position of this thread's row in work item itx
      const ConvItem it = conv_item(p, cta + itx * nctas);
      const int pos = it.mt * 128 + row;
      pvalid = pos < p.P;
      const int n = pvalid ? pos / p.OHW : 0, r = pos - n * p.OHW, oh = r / p.OW, ow = r - oh * p.OW;
      ih0 = oh * p.stride - p.pad_h;
      iw0 = ow * p.stride - p.pad_w;
      xn = p.x[it.prob] + (int64_t)n * p.Cin * p.IHW;
    };
    if (total > 0) locate();

    // gathers this thread's 16 values of the cursor's box into ring slot `slot`, then advances the cursor
    auto issue = [&](int slot) {
      const uint32_t dst = ring + (uint32_t)slot * 16384u;
      if (!p.flat) {
        const int ih = ih0 + kh, iw = iw0 + kw;
        const bool ok = pvalid && (unsigned)ih < (unsigned)p.IH && (unsigned)iw < (unsigned)p.IW;
        const float *src = ok ? xn + (int64_t)(cb * 32 + hsel * 16) * p.IHW + ih * p.IW + iw : xn;
        const uint32_t cs = ok ? (uint32_t)p.IHW : 0u, ign = ok ? 0u : 1u;
#pragma unroll
        for (int c = 0; c < 16; ++c) cp_async4(dst + c * 512, src + (uint32_t)c * cs, ign);
      } else {
        // flat form: this thread's 16 k are 16 >> lg kernel rows of KWP = 1 << lg taps each; a row's (channel, kh)
        // comes from the table once, its taps are consecutive addresses
        const int row0 = (cb * 32 + hsel * 16) >> p.flat_lg;
        const float *origin = xn + ih0 * p.IW + iw0;
        switch (p.flat_lg) {
          case 0: flat_rows<0>(ktab + row0, origin, xn, dst, pvalid, ih0, iw0, p.IH, p.IW, p.KW); break;
          case 1: flat_rows<1>(ktab + row0, origin, xn, dst, pvalid, ih0, iw0, p.IH, p.IW, p.KW); break;
          case 2: flat_rows<2>(ktab + row0, origin, xn, dst, pvalid, ih0, iw0, p.IH, p.IW, p.KW); break;
          case 3: flat_rows<3>(ktab + row0, origin, xn, dst, pvalid, ih0, iw0, p.IH, p.IW, p.KW); break;
          default: flat_rows<4>(ktab + row0, origin, xn, dst, pvalid, ih0, iw0, p.IH, p.IW, p.KW); break;
        }
      }
      if (++kw == kw_n) {
        kw = 0;
        if (++kh == kh_n) {
          kh = 0;
          if (++cb == cb_n) {
            cb = 0;
            ++itx;
            if (itx < my_items) locate();
          }
        }
      }
    };

    int slot_in = 0;
#pragma unroll 1
    for (int j = 0; j < kARing - 1; ++j) {
      if (j < total && !(DBG && p.debug & 1)) issue(slot_in);
      cp_async_commit();
      if (++slot_in == kARing) slot_in = 0;
    }
    int slot_out = 0;
#pragma unroll 1
    for (int i = 0; i < total; ++i) {
      if (i + kARing - 1 < total && !(DBG && p.debug & 1)) issue(slot_in);
      cp_async_commit();
      if (++slot_in == kARing) slot_in = 0;
      cp_async_wait<kARing - 1>();  // this thread's copies of box i have landed
      uint32_t v[16];
#pragma unroll
      for (int c = 0; c < 16; ++c)
        asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v[c]) : "r"(ring + (uint32_t)slot_out * 16384u + c * 512u) : "memory");
      if (++slot_out == kARing) slot_out = 0;
      const uint32_t s = (uint32_t)i & (kConvStages - 1), ph = ((uint32_t)i / kConvStages) & 1u;
      const bool tr = DBG && p.trace && cta == 0 && warp == 2 && lane == 0 && i < 512;
      a32_wait_wd(bar_empty + 8 * s, ph ^ 1u);
      tc_fence_after();
      // hi = rna_tf32(x), lo = rna_tf32(x - hi) with integer rounding: add half a tf32 ulp, clear the 13 low bits
      // (for lo the tensor core's own truncation of the operand does the clearing, as in gram_tma.cu)
      uint32_t hi[16];
#pragma unroll
      for (int c = 0; c < 16; ++c) hi[c] = (v[c] + 0x1000u) & 0xffffe000u;
      tmem_st16(a_base + s * 64, hi);
#pragma unroll
      for (int c = 0; c < 16; ++c)
        hi[c] = __float_as_uint(__uint_as_float(v[c]) - __uint_as_float(hi[c])) + 0x1000u;  // the core drops the low bits
      tmem_st16(a_base + s * 64 + 32, hi);
      tmem_st_wait();
      if (tr) p.trace[i * 16 + 3] = clock64();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) a32_arrive(bar_full + 8 * s);
    }
  } else {
    // ------------------------------------------------------------------ promotion / epilogue
    constexpr int COLS = TN / 2;
    const int q = warp & 3;
    const int half = (warp - 10) >> 2;
    uint32_t chain = 0;
    for (int item = cta; item < p.total_items; item += nctas) {
      const ConvItem it = conv_item(p, item);
      // promotion accumulators as fp32 pairs: one add.rn.f32x2 per two columns halves the issue slots this role
      // takes from the MMA-issuing warp's scheduler
      unsigned long long acc2[COLS / 2];
#pragma unroll
      for (int c = 0; c < COLS / 2; ++c) acc2[c] = 0ull;
      for (int b0 = 0; b0 < p.nbox; b0 += CH, ++chain) {
        const uint32_t buf = chain & 1u;
        a32_wait_wd(bar_acc_full + 8 * buf, (chain >> 1) & 1u);
        const bool tr = DBG && p.trace && cta == 0 && warp == 10 && lane == 0 && chain < 512;
        if (tr) p.trace[chain * 16 + 5] = clock64();
        tc_fence_after();
        const uint32_t t0 = tmem_base + ((uint32_t)(q * 32) << 16) + buf * TN + half * COLS;
#pragma unroll
        for (int c = 0; c < COLS / 16; ++c) {
          uint32_t v[16];
          tmem_ld16(t0 + c * 16, v);
          tmem_ld_wait();
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            unsigned long long pr;
            asm("mov.b64 %0, {%1, %2};" : "=l"(pr) : "r"(v[2 * e]), "r"(v[2 * e + 1]));
            asm("add.rn.f32x2 %0, %0, %1;" : "+l"(acc2[c * 8 + e]) : "l"(pr));
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) a32_arrive(bar_acc_empty + 8 * buf);
        if (tr) p.trace[chain * 16 + 7] = clock64();
      }
      float acc[COLS];
#pragma unroll
      for (int c = 0; c < COLS / 2; ++c) {
        uint32_t lo, hi;
        asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(acc2[c]));
        acc[2 * c] = __uint_as_float(lo);
        acc[2 * c + 1] = __uint_as_float(hi);
      }
      const int pos = it.mt * 128 + q * 32 + lane;
      if (pos < p.P && !(DBG && p.debug & 4)) {
        const int n = pos / p.OHW, r = pos - n * p.OHW;
        const int co0 = it.nt * TN + half * COLS;
        float *o = p.out[it.prob] + ((int64_t)n * p.Cout + co0) * p.OHW + r;
        const float *bias = p.bias[it.prob];
        const int ohw = p.OHW;
        const int nc = min(COLS, p.Cout - co0);
        float *o2 = p.out2[it.prob] ? p.out2[it.prob] + ((int64_t)n * p.Cout + co0) * p.OHW + r : nullptr;
        const float2 *ss = p.post[it.prob] ? p.post[it.prob] + co0 : nullptr;
        const bool relu = p.post_relu != 0;
        // one IMAD.WIDE + one STG per value on the common paths (full channel tile): the store loop is what bounds
        // the small-K layers, 64 values per thread and item.  The fused eval-mode BatchNorm (+ ReLU) behind the
        // convolution is a second output from the same registers instead of two more passes over the activation.
        if (nc == COLS && bias == nullptr && o2 == nullptr) {
          store_tile<COLS, false, false>(acc, o, o2, ohw, bias, ss, relu, nc);
        } else if (nc == COLS && bias == nullptr) {
          store_tile<COLS, false, true>(acc, o, o2, ohw, bias, ss, relu, nc);
        } else {
          store_tile_ragged<COLS>(acc, o, o2, ohw, bias ? bias + co0 : nullptr, ss, relu, nc);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// w[Cout][Cin][KH][KW] -> hi / lo planes [2][taps][Cout][Kc] (include/pleas_b200.h)
__global__ void conv_pack_weights_kernel(const float *__restrict__ w, float *__restrict__ packed, int Cout, int Cin,
                                         int KH, int KW, int taps, int Kc, int flat, int flat_lg) {
  const int64_t plane = (int64_t)taps * Cout * Kc;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < plane; idx += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(idx % Kc);
    const int co = (int)((idx / Kc) % Cout);
    const int t = (int)(idx / ((int64_t)Kc * Cout));
    float v = 0.f;
    if (!flat) {
      v = w[((int64_t)co * Cin + k) * (KH * KW) + t];
    } else {
      const int g = k >> flat_lg, kw = k & ((1 << flat_lg) - 1);  // kernel row (ci, kh) and tap inside it
      if (g < Cin * KH && kw < KW) v = w[((int64_t)co * Cin * KH + g) * KW + kw];
    }
    const float hi = to_tf32(v);
    packed[idx] = hi;
    packed[plane + idx] = to_tf32(v - hi);
  }
}

static unsigned long long *g_conv_trace = nullptr;

struct ConvGeometry {
  int flat, taps, Kc, flat_lg;
};
static ConvGeometry conv_geometry(int64_t Cin, int KH, int KW) {
  ConvGeometry g;
  g.flat = (Cin % 32) != 0;
  g.taps = g.flat ? 1 : KH * KW;
  g.flat_lg = 0;
  while ((1 << g.flat_lg) < KW) ++g.flat_lg;  // kernel rows padded to a power of two of taps (zero weights)
  g.Kc = g.flat ? (int)(ceil_div((Cin * KH) << g.flat_lg, 32) * 32) : (int)Cin;
  return g;
}

static int make_weight_map(CUtensorMap *m, const float *packed, int64_t Cout, const ConvGeometry &g, int tn) {
  EncodeTiledFn enc = encode_tiled();
  PLB_REQUIRE(enc != nullptr, PLB_EINVAL, "plb_conv2d_forward: cuTensorMapEncodeTiled is not available from this driver");
  cuuint64_t gdim[4] = {(cuuint64_t)g.Kc, (cuuint64_t)Cout, (cuuint64_t)g.taps, 2};
  cuuint64_t gstride[3] = {(cuuint64_t)g.Kc * 4, (cuuint64_t)g.Kc * Cout * 4, (cuuint64_t)g.Kc * Cout * g.taps * 4};
  cuuint32_t box[4] = {32, (cuuint32_t)tn, 1, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void *)packed, gdim, gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PLB_REQUIRE(r == CUDA_SUCCESS, PLB_EINVAL, "plb_conv2d_forward: cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return PLB_OK;
}

template <int TN, int CH, bool DBG>
static int launch_conv(const CUtensorMap &m0, const CUtensorMap &m1, const ConvParams &p, cudaStream_t stream) {
  constexpr int smem_bytes = ConvCfg<TN>::kSmemBytes;
  if (int rc = ensure_dynamic_smem((const void *)conv3xtf32_kernel<TN, CH, DBG>, smem_bytes, "conv3xtf32_kernel"))
    return rc;
  const int grid = min(p.total_items, device_sm_count());
  conv3xtf32_kernel<TN, CH, DBG><<<grid, kConvThreads, smem_bytes, stream>>>(m0, m1, p);
  return launch_status("conv3xtf32_kernel");
}

}  // namespace plb

// experiments only: CTA 0 of every later plb_conv2d_forward launch writes 8 clock64 stamps per box (first 512 boxes)
// [TMA issue, loader data ready, loader slot free, loader stored, MMA sees A, MMA sees B, MMA issued, -]
extern "C" int plb_conv_debug_set_trace(unsigned long long *dev_buf) {
  plb::g_conv_trace = dev_buf;
  return PLB_OK;
}

extern "C" int64_t plb_conv_packed_floats(int64_t Cout, int64_t Cin, int32_t KH, int32_t KW) {
  if (Cout <= 0 || Cin <= 0 || KH <= 0 || KW <= 0) return 0;
  const plb::ConvGeometry g = plb::conv_geometry(Cin, KH, KW);
  return 2ll * g.taps * Cout * g.Kc;
}

extern "C" int plb_conv_pack_weights(const float *w, int64_t Cout, int64_t Cin, int32_t KH, int32_t KW, float *packed,
                                     void *stream) {
  using namespace plb;
  PLB_REQUIRE(w && packed, PLB_EINVAL, "plb_conv_pack_weights: null pointer");
  PLB_REQUIRE(Cout > 0 && Cin > 0 && KH > 0 && KW > 0, PLB_EINVAL, "plb_conv_pack_weights: empty weight");
  const ConvGeometry g = conv_geometry(Cin, KH, KW);
  PLB_REQUIRE(!g.flat || KW <= 16, PLB_ESIZE, "plb_conv_pack_weights: Cin %% 32 != 0 needs KW <= 16");
  PLB_REQUIRE(!g.flat || g.Kc <= kConvMaxFlatK, PLB_ESIZE,
              "plb_conv_pack_weights: Cin %% 32 != 0 needs Cin*KH*pow2(KW) <= %d", kConvMaxFlatK);
  const int64_t plane = (int64_t)g.taps * Cout * g.Kc;
  PLB_REQUIRE(plane < (1ll << 31), PLB_ESIZE, "plb_conv_pack_weights: weight too large");
  const int64_t want = ceil_div(plane, 256);
  const int blocks = (int)(want < 148 * 8 ? want : 148 * 8);
  conv_pack_weights_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(w, packed, (int)Cout, (int)Cin, KH, KW, g.taps,
                                                                     g.Kc, g.flat, g.flat_lg);
  return launch_status("conv_pack_weights_kernel");
}

extern "C" int plb_conv2d_forward(const float *const *x, const float *const *packed_w, const float *const *bias,
                                  float *const *out, int32_t nprob, int64_t NB, int64_t Cin, int64_t IH, int64_t IW,
                                  int64_t Cout, int32_t KH, int32_t KW, int32_t stride, int32_t pad_h, int32_t pad_w,
                                  void *stream) {
  return plb_conv2d_affine_forward(x, packed_w, bias, out, nullptr, nullptr, 0, nprob, NB, Cin, IH, IW, Cout, KH, KW,
                                   stride, pad_h, pad_w, stream);
}

extern "C" int plb_conv2d_affine_forward(const float *const *x, const float *const *packed_w,
                                         const float *const *bias, float *const *out,
                                         const float *const *scale_shift, float *const *out2, int32_t relu,
                                         int32_t nprob, int64_t NB, int64_t Cin, int64_t IH, int64_t IW, int64_t Cout,
                                         int32_t KH, int32_t KW, int32_t stride, int32_t pad_h, int32_t pad_w,
                                         void *stream) {
  using namespace plb;
  PLB_REQUIRE(x && packed_w && out, PLB_EINVAL, "plb_conv2d_forward: null pointer table");
  PLB_REQUIRE(nprob == 1 || nprob == 2, PLB_EINVAL, "plb_conv2d_forward: one or two problems per launch");
  PLB_REQUIRE(NB > 0 && Cin > 0 && IH > 0 && IW > 0 && Cout > 0 && KH > 0 && KW > 0 && stride > 0 && pad_h >= 0 &&
                  pad_w >= 0,
              PLB_EINVAL, "plb_conv2d_forward: bad geometry");
  const int64_t OH = (IH + 2 * pad_h - KH) / stride + 1, OW = (IW + 2 * pad_w - KW) / stride + 1;
  PLB_REQUIRE(OH > 0 && OW > 0, PLB_EINVAL, "plb_conv2d_forward: empty output");
  PLB_REQUIRE(NB * OH * OW < (1ll << 31) - 128 && NB * Cin * IH * IW < (1ll << 40) && Cin * IH * IW < (1ll << 31) &&
                  KH < 256 && KW < 256,
              PLB_ESIZE, "plb_conv2d_forward: extent too large");
  const ConvGeometry g = conv_geometry(Cin, KH, KW);
  PLB_REQUIRE(!g.flat || KW <= 16, PLB_ESIZE, "plb_conv2d_forward: Cin %% 32 != 0 needs KW <= 16");
  PLB_REQUIRE(!g.flat || g.Kc <= kConvMaxFlatK, PLB_ESIZE,
              "plb_conv2d_forward: Cin %% 32 != 0 needs Cin*KH*pow2(KW) <= %d", kConvMaxFlatK);
  ConvParams p = {};
  for (int i = 0; i < nprob; ++i) {
    PLB_REQUIRE(x[i] && packed_w[i] && out[i], PLB_EINVAL, "plb_conv2d_forward: null pointer");
    PLB_REQUIRE(((uintptr_t)packed_w[i] & 15) == 0, PLB_EALIGN, "plb_conv2d_forward: packed weights must be 16-byte aligned");
    p.x[i] = x[i];
    p.out[i] = out[i];
    p.bias[i] = bias ? bias[i] : nullptr;
    PLB_REQUIRE((scale_shift == nullptr) == (out2 == nullptr) &&
                    (out2 == nullptr || ((scale_shift[i] != nullptr) && (out2[i] != nullptr))),
                PLB_EINVAL, "plb_conv2d_affine_forward: scale_shift and out2 go together");
    PLB_REQUIRE(scale_shift == nullptr || ((uintptr_t)scale_shift[i] & 7) == 0, PLB_EALIGN,
                "plb_conv2d_affine_forward: scale_shift must be 8-byte aligned");
    p.post[i] = scale_shift ? reinterpret_cast<const float2 *>(scale_shift[i]) : nullptr;
    p.out2[i] = out2 ? out2[i] : nullptr;
  }
  p.nprob = nprob;
  p.post_relu = relu;
  p.NB = (int)NB, p.Cin = (int)Cin, p.IH = (int)IH, p.IW = (int)IW, p.Cout = (int)Cout, p.OH = (int)OH, p.OW = (int)OW;
  p.KH = KH, p.KW = KW, p.stride = stride, p.pad_h = pad_h, p.pad_w = pad_w;
  p.P = (int)(NB * OH * OW), p.OHW = (int)(OH * OW), p.IHW = (int)(IH * IW);
  p.flat = g.flat, p.taps = g.taps, p.flat_groups = (int)(Cin * KH), p.flat_lg = g.flat_lg;
  p.nbox = g.taps * (g.Kc / 32);
  static int debug = -1;
  if (debug < 0) {
    const char *d = getenv("PLB_CONV_DEBUG");
    debug = d ? atoi(d) : 0;
  }
  p.debug = debug;
  p.trace = g_conv_trace;
  // The tensor core truncates when it adds into its fp32 accumulator (about -1e-7 relative per 16 k, gemm.cu): a
  // bias that compounds through the layers of a network (activations shrink a little in every layer).  Chains are
  // therefore TWO boxes (64 k), each chain's lo x hi products are issued before its hi x hi ones (they add at 2^-11
  // of the final magnitude, so their truncation costs nothing), and the promotion warps add every chain with
  // round-to-nearest.  Measured on the ResNet-50 pair (tests/test_configs_gpu.py, worst deviation of a group's
  // objective from the reference's; profiles/r02_notes.md): 8-box chains in k order > 1.3e-5, 2 boxes in k order
  // 1.0e-5, 1 box 5.2e-6, 2 boxes small products first 4.2e-6 (cuDNN fp32 forwards: ~4e-6).
  static int chain = 0;
  if (chain == 0) {
    const char *c = getenv("PLB_CONV_CHAIN");  // experiments: boxes per accumulation chain
    chain = (c && atoi(c) > 0 && atoi(c) <= kConvStages / 2) ? atoi(c) : 2;
  }
  p.chain_boxes = chain;
  const int tn = Cout <= 64 ? 64 : 128;
  p.m_tiles = (int)ceil_div(p.P, 128);
  p.n_tiles = (int)ceil_div(Cout, tn);
  const int64_t items = (int64_t)p.m_tiles * p.n_tiles * nprob;
  PLB_REQUIRE(items * p.nbox < (1ll << 31), PLB_ESIZE, "plb_conv2d_forward: too many work items");
  p.total_items = (int)items;
  CUtensorMap m0, m1;
  if (int rc = make_weight_map(&m0, packed_w[0], Cout, g, tn)) return rc;
  if (int rc = make_weight_map(&m1, packed_w[nprob - 1], Cout, g, tn)) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const bool dbg = p.debug != 0 || p.trace != nullptr;
  if (dbg || chain != 2) {  // experiments: runtime switches compiled in
    if (chain == 1) return tn == 64 ? launch_conv<64, 1, true>(m0, m1, p, s) : launch_conv<128, 1, true>(m0, m1, p, s);
    return tn == 64 ? launch_conv<64, 2, true>(m0, m1, p, s) : launch_conv<128, 2, true>(m0, m1, p, s);
  }
  return tn == 64 ? launch_conv<64, 2, false>(m0, m1, p, s) : launch_conv<128, 2, false>(m0, m1, p, s);
}
