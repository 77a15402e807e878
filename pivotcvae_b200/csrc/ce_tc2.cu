// ce_tc2.cu — full-catalog soft-max cross-entropy with BOTH contractions on the tensor cores
// (engine PCV_CE_ENGINE_TF32 of pcv_ce_fwd_bwd / pcv_ce_partials; dense mask, D = 8, 16, 32, 64 or 128).
//
// Replaces pivotcvae.py:274 (p = mm(prox, table.t())) + train_generative.py:59 (CrossEntropyLoss) and their
// backward, like ce.cu.  ce_tc.cu (the first tensor-core engine) computed the logits with tcgen05 but accumulated
// d loss / d q = sum_j softmax_j w_j with 8 FFMA per logit on the CUDA cores: FMA-pipe-bound at ~23 cycles per 32
// logits per scheduler.  Here the gradient is a second MMA, flash-attention style (BN items per tile, see Ce2Cfg):
//
//   S[128 x BN]  = Q[128 x D] . W_tile^T                     D/8 accumulating tcgen05.mma kind::tf32 (K = 8 each),
//                                                            A/B from shared memory
//   P            = exp(S - c_row)                            epilogue warps: TMEM -> registers -> TMEM (in place)
//   dq[128 x NG] += P[128 x BN] . Wt_tile^T                  tcgen05.mma, A = P from TENSOR MEMORY, B = the
//                                                            transposed tile [NG x BN items], NG = max(D, 16)
//                                                            (D = 8: 8 dims + 8 zero rows, as M = 128 needs N >= 16)
//
// so an epilogue thread spends 3 instructions per logit (FFMA, MUFU.EX2, FADD) instead of 13, at every D.  Measured at
// C3, D = 8 (100 k items x 20480 rows): 0.70 ms vs 1.41 ms for ce_tc.cu; the MUFU pipe (one ex2 per logit, 16 / clk /
// SM) would allow 0.44 ms — what is left is the single MMA-issuing warp (17 tcgen05.mma per 128-item tile, see
// umma_*_elect).  Larger D adds score MMAs per tile and streams D times more table bytes (W and its transposed image)
// per tile; see DESIGN §5 for the measured times per D.  There is no running maximum to rescale the TMEM accumulator
// by: every row uses a FIXED reference exponent c_row chosen by ce_ref_kernel from rigorous bounds —
//   s_j <= ub = |q| max|w| (Cauchy-Schwarz),   lb = max(target logit, logits of the first 32 items) <= max_j s_j,
//   c = max(lb, ub - 60)   =>   s_j - c <= 60 (no overflow: e^60 * N << 3e38) and max_j s_j - c >= lb - ub + 60,
// which cannot underflow when lb >= ub - 140.  None of this depends on D.  Rows that fail that test (never seen in
// practice: it needs |q| max|w| > 70 with a far-off target) are flagged and redone exactly by ce_rowfix_kernel.
// The per-(split, row) records (c, l, count, acc[D]) have the layout of ce.cu and are merged by the same
// ce_finalize_kernel (target logit re-derived with the exact fp32 FMA chain).
#include <mutex>

#include "table_images.cuh"

namespace pcv {

constexpr int C2_BUFS = 3;                      // S/P buffers in flight
constexpr int C2_EPI_WARPS = 16;                // 4 per TMEM lane quarter, each a BN/2-column half of every other tile
constexpr int C2_THREADS = 64 + 32 * C2_EPI_WARPS;

// Per-D tile shapes.  Shared memory = STAGES x (W + Wt tile) + A_BUFS query tiles <= 227 KB; TMEM = 3 S/P buffers of BN
// columns + DQ_ACCS gradient accumulators of NG columns <= 512.  STAGES >= 3: a stage is released by the gradient MMA
// of its tile, which is issued two tiles after the score MMA (so stage t % STAGES must not wait on tile t - 2).
//   D     BN   W + Wt per stage   stages   query tile x buffers   dq accumulators
//   8    128    4 +  8 KB           12        4 KB x 2              4 x 16
//   16   128    8 +  8 KB           10        8 KB x 2              4 x 16
//   32   128   16 + 16 KB            5       16 KB x 2              2 x 32
//   64    64   16 + 16 KB            4       32 KB x 2              2 x 64
//   128   32   16 + 16 KB            4       64 KB x 1              2 x 128
template <int D>
struct Ce2Cfg {
  static constexpr int KA = D / 8;                                 // k-atoms (8 fp32 = 32 B) of an embedding row
  static constexpr int BN = WtGeom<D>::BN;                         // items per tile (= TMEM columns of one S/P buffer)
  static constexpr int NG = WtGeom<D>::NG;                         // N of the gradient MMA
  static constexpr int STAGES = D == 8 ? 12 : D == 16 ? 10 : D == 32 ? 5 : 4;
  static constexpr int A_BUFS = D <= 64 ? 2 : 1;
  // N = 16 gradient MMAs are 8 cycles of work each: four independent accumulators keep the tensor pipe from waiting on
  // its own accumulate latency; wider ones need fewer
  static constexpr int DQ_ACCS = D <= 16 ? 4 : 2;
  static constexpr int DQ_COL = (C2_BUFS * BN + NG - 1) / NG * NG;   // first dq accumulator column
  static constexpr int W_FLOATS = BN * D;        // W tile: KA k-atoms of [BN rows x 32 B] (SWIZZLE_32B image)
  static constexpr int WT_FLOATS = BN * NG;      // transposed tile: BN / 8 k-atoms of [NG rows x 32 B]
  static constexpr int A_FLOATS = TC_BM * D;     // query tile: KA k-atoms of [128 rows x 32 B]
  static constexpr int HALF = BN / 2;            // columns of a tile one epilogue warp exponentiates
  static constexpr int CW = HALF < 32 ? HALF : 32;   // ... in chunks of CW columns
  static constexpr int NCH = HALF / CW;
  static constexpr int GW = D < 32 ? D : 32;     // dq columns read out per TMEM load
  static constexpr int REC = 3 + D;
  static_assert(STAGES >= 3, "see above");
  static_assert(NCH == 1 || NCH == 2, "one or two epilogue chunks per tile half");
  static_assert(DQ_COL + DQ_ACCS * NG <= 512, "TMEM columns");
};

template <int D>
struct __align__(1024) Ce2Smem {
  using C = Ce2Cfg<D>;
  float w[C::STAGES][C::W_FLOATS];
  float wt[C::STAGES][C::WT_FLOATS];
  float a[C::A_BUFS][C::A_FLOATS];
  unsigned long long full[C::STAGES], empty[C::STAGES], tfull[C2_BUFS], pfull[C2_BUFS], tempty[C2_BUFS];
  unsigned long long afull[C::A_BUFS], aempty[C::A_BUFS], dqfull, dqempty;
  float lsum[2][3][TC_BM];   // per-row l of the column slices 1..3 of a work item (double-buffered by item parity)
  uint32_t tmem_base;
};

// kind::tf32, fp32 accumulate, K-major operands, M = 128: N = BN (scores) / N = NG (gradient)
template <int N>
constexpr uint32_t C2_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);

// D[tmem] (+)= A[tmem] . B[smem]^T : the A operand is read from tensor memory (lane = row, one 32-bit column per k)
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}

// (the MMA warp runs converged: see umma_tf32_elect in tc_common.cuh)
__device__ __forceinline__ void umma_tf32_ts_elect(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p, q;\n"
      "elect.sync _|q, 0xffffffff;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
#define C2_ST32(taddr, v)                                                                                   \
  asm volatile(                                                                                             \
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "                                                       \
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "                            \
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"                    \
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),  \
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),        \
        "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),      \
        "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])       \
      : "memory")

// 16-column forms (the half-tiles of D = 128) and the 8- / 16-column dq read-out of D = 8 / 16
#define C2_LD16(v, taddr)                                                                                   \
  asm volatile(                                                                                             \
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "                                                             \
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"                      \
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),     \
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]) \
      : "r"(taddr))
#define C2_WAIT_LD16(v)                                                                                     \
  asm volatile("tcgen05.wait::ld.sync.aligned;"                                                             \
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]),        \
                 "+r"(v[7]), "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]),    \
                 "+r"(v[14]), "+r"(v[15])::"memory")
#define C2_ST16(taddr, v)                                                                                   \
  asm volatile(                                                                                             \
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "                                                       \
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"                            \
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),  \
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])         \
      : "memory")
#define C2_LD8(v, taddr)                                                                                    \
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"              \
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) \
               : "r"(taddr))
#define C2_WAIT_LD8(v)                                                                                      \
  asm volatile("tcgen05.wait::ld.sync.aligned;"                                                             \
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]),        \
                 "+r"(v[7])::"memory")

// n-column TMEM load / wait / store of this warp's lane quarter (n = 8, 16 or 32)
template <int n>
__device__ __forceinline__ void c2_ld(uint32_t (&v)[n], uint32_t taddr) {
  if constexpr (n == 32) TC_LD32(v, taddr);
  else if constexpr (n == 16) C2_LD16(v, taddr);
  else C2_LD8(v, taddr);
}
template <int n>
__device__ __forceinline__ void c2_wait_ld(uint32_t (&v)[n]) {
  if constexpr (n == 32) TC_WAIT_LD(v);
  else if constexpr (n == 16) C2_WAIT_LD16(v);
  else C2_WAIT_LD8(v);
}
template <int n>
__device__ __forceinline__ void c2_st(uint32_t taddr, uint32_t (&v)[n]) {
  static_assert(n == 32 || n == 16, "P chunks are 16 or 32 columns");
  if constexpr (n == 32) C2_ST32(taddr, v);
  else C2_ST16(taddr, v);
}

__device__ __forceinline__ float c2_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// sequential-k fp32 FMA chain over D (the order the rest of the library uses for a logit)
template <int D>
__device__ __forceinline__ float c2_dot(const float *__restrict__ q, const float *__restrict__ w) {
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < D; k += 4) {
    const float4 q4 = __ldg(reinterpret_cast<const float4 *>(q + k));
    const float4 w4 = __ldg(reinterpret_cast<const float4 *>(w + k));
    s = fmaf(q4.x, w4.x, s); s = fmaf(q4.y, w4.y, s); s = fmaf(q4.z, w4.z, s); s = fmaf(q4.w, w4.w, s);
  }
  return s;
}

// ---- per-row reference exponent + safety flag (see the header)
template <int D>
__global__ void __launch_bounds__(256)
ce_ref_kernel(const float *__restrict__ W, int64_t n_rows, int64_t row_offset, const float *__restrict__ max_row_norm,
              const float *__restrict__ Q,
              const int64_t *__restrict__ targets, int64_t M, float *__restrict__ cref, unsigned char *__restrict__ unsafe) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const float *q = Q + row * D;
  float lb = (lane < n_rows) ? c2_dot<D>(q, W + (int64_t)lane * D) : -INFINITY;   // lane = one of the first 32 items
  const int64_t t = targets[row] - row_offset;
  if (lane == 0 && t >= 0 && t < n_rows) lb = fmaxf(lb, c2_dot<D>(q, W + t * D));
  lb = warp_max(lb);
  if (lane == 0) {
    const float ss = c2_dot<D>(q, q);
    const float ub = sqrtf(ss) * __ldg(max_row_norm) * 1.01f + 1e-30f;   // >= every tf32 logit (truncation only shrinks |s|)
    lb -= 0.01f * ub;                                              // the tf32 logit of that item may sit a little lower
    const bool ok = lb >= ub - 140.f && ub < 1.0e30f;
    cref[row] = ok ? fmaxf(lb, ub - 60.f) : 0.f;
    unsafe[row] = ok ? 0 : 1;
  }
}

// ---- exact redo of a flagged row over this table shard (one warp per row; normally every warp exits at once):
// stream 0 of the row gets the exact partial (running max m, l, acc), every other stream an empty record.  The
// gradient is accumulated in chunks of at most 32 dimensions, one online pass over the shard per chunk (m and l come
// out of every pass identical; the last pass's are kept), so no lane holds more than 32 accumulators.
template <int D>
__global__ void __launch_bounds__(256)
ce_rowfix_kernel(const float *__restrict__ W, int64_t n_rows, const float *__restrict__ Q, int64_t M,
                 const unsigned char *__restrict__ unsafe, int n_streams, float *__restrict__ part) {
  constexpr int CK = D < 32 ? D : 32;
  constexpr int REC = 3 + D;
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M || !unsafe[row]) return;
  const float *q = Q + row * D;
  for (int k0 = 0; k0 < D; k0 += CK) {
    float m = -INFINITY, l = 0.f, acc[CK];
#pragma unroll
    for (int k = 0; k < CK; ++k) acc[k] = 0.f;
    for (int64_t j = lane; j < n_rows; j += 32) {
      const float *w = W + j * D;
      const float s = c2_dot<D>(q, w);
      if (s > m) {
        const float sc = __expf(m - s);
        l *= sc;
#pragma unroll
        for (int k = 0; k < CK; ++k) acc[k] *= sc;
        m = s;
      }
      const float p = __expf(s - m);
      l += p;
#pragma unroll
      for (int k = 0; k < CK; ++k) acc[k] = fmaf(p, __ldg(w + k0 + k), acc[k]);
    }
    const float mw = warp_max(m);
    const float sc = (m == -INFINITY) ? 0.f : __expf(m - mw);
    l = warp_sum(l * sc);
#pragma unroll
    for (int k = 0; k < CK; ++k) acc[k] = warp_sum(acc[k] * sc);
    if (lane == 0) {
      for (int s = 0; s < n_streams; ++s) {
        float *rec = part + ((int64_t)s * M + row) * REC;
        if (k0 + CK == D) {
          rec[0] = s == 0 ? mw : -INFINITY;
          rec[1] = s == 0 ? l : 0.f;
          rec[2] = __int_as_float(s == 0 ? (int)n_rows : 0);
        }
#pragma unroll
        for (int k = 0; k < CK; ++k) rec[3 + k0 + k] = s == 0 ? acc[k] : 0.f;
      }
    }
  }
}

// Transposed, pre-swizzled image of the table for the gradient MMA's B operand (layout: wt_index).  The buffer is
// zero-filled first (padding rows, tail of the last tile).  One thread per table element.
template <int D>
__global__ void pack_wt_kernel(const float *__restrict__ W, int64_t n_rows, float *__restrict__ out) {
  const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n_rows * D) return;
  out[wt_index<D>(f / D, (int)(f % D))] = W[f];
}

// 18 warps on the 4 SM sub-partitions (16 K registers each, five warps on two of them) allow 96 registers a thread
template <int D>
__global__ void __launch_bounds__(C2_THREADS, 1)
ce_tc2_kernel(const float *__restrict__ Wsw, const float *__restrict__ Wt, int64_t n_rows, const float *__restrict__ Q, int64_t M,
              const float *__restrict__ cref, int64_t items_per_split, int n_split, int n_work, float *__restrict__ part) {
  using C = Ce2Cfg<D>;
  constexpr int BN = C::BN, KA = C::KA, NG = C::NG, STAGES = C::STAGES, A_BUFS = C::A_BUFS, DQ_ACCS = C::DQ_ACCS;
  constexpr int HALF = C::HALF, CW = C::CW, NCH = C::NCH, GW = C::GW;
  constexpr uint32_t IDESC_S = C2_IDESC<BN>, IDESC_G = C2_IDESC<NG>;
  extern __shared__ unsigned char smem_raw[];
  Ce2Smem<D> &S = *reinterpret_cast<Ce2Smem<D> *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int lane = threadIdx.x & 31;
  // roles: hardware warps 0..15 = epilogue, 16 = producer, 17 = MMA issuer.  The scheduler arbitrates highest warp id
  // first, so the two single-thread control warps are never starved by the MUFU-bound epilogue warps of their
  // sub-partition.  (`warp` keeps the logical numbering used below: 0 = producer, 1 = MMA, 2.. = epilogue.)
  const int hw_warp = threadIdx.x >> 5;
  const int warp = hw_warp >= C2_EPI_WARPS ? hw_warp - C2_EPI_WARPS : hw_warp + 2;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&S.full[s], 1); mbar_init(&S.empty[s], 1); }
    for (int b = 0; b < C2_BUFS; ++b) {
      mbar_init(&S.tfull[b], 1); mbar_init(&S.pfull[b], C2_EPI_WARPS / 2); mbar_init(&S.tempty[b], 1);
    }
    for (int b = 0; b < A_BUFS; ++b) { mbar_init(&S.afull[b], 1); mbar_init(&S.aempty[b], 1); }
    mbar_init(&S.dqfull, 1);
    mbar_init(&S.dqempty, 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&S.tmem_base)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = S.tmem_base;

  const int w_begin = (int)((int64_t)blockIdx.x * n_work / gridDim.x);
  const int w_end = (int)((int64_t)(blockIdx.x + 1) * n_work / gridDim.x);
  auto item_rows = [&](int w) { return (int64_t)(w / n_split) * TC_BM; };
  auto item_split = [&](int w) { return (w % n_split + (w / n_split) * 3) % n_split; };
  auto item_jb = [&](int w) { return (int64_t)item_split(w) * items_per_split; };
  auto item_tiles = [&](int w) {
    const int64_t jb = item_jb(w), je = min(n_rows, jb + items_per_split);
    return (int)((je - jb + BN - 1) / BN);
  };

  if (warp == 0) {
    // ---------------- producer: query tile of the work item, then its W / Wt tiles ----------------
    uint32_t gt = 0;
    int it = 0;
    for (int w = w_begin; w < w_end; ++w, ++it) {
      const int ab = it % A_BUFS;
      mbar_wait(&S.aempty[ab], ((it / A_BUFS) & 1) ^ 1);
      {
        // 128 query rows per k-atom: row t at byte t*32, 16-byte chunk c at ((c ^ bit2(t)) * 16)  (SWIZZLE_32B image)
        const int64_t row_base = item_rows(w);
#pragma unroll
        for (int i = 0; i < TC_BM / 32; ++i) {
          const int t = lane + 32 * i;
          const int64_t row = row_base + t;
          const int sw = (t >> 2) & 1;
#pragma unroll 4
          for (int a = 0; a < KA; ++a) {
            float4 q0 = make_float4(0.f, 0.f, 0.f, 0.f), q1 = q0;
            if (row < M) {
              q0 = __ldg(reinterpret_cast<const float4 *>(Q + row * D + a * 8));
              q1 = __ldg(reinterpret_cast<const float4 *>(Q + row * D + a * 8) + 1);
            }
            float4 *dst = reinterpret_cast<float4 *>(S.a[ab] + a * (TC_BM * 8) + t * 8);
            dst[0 ^ sw] = q0;
            dst[1 ^ sw] = q1;
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&S.afull[ab]);
      }
      if (lane == 0) {
        const int64_t j_begin = item_jb(w);
        const int n_tiles = item_tiles(w);
        for (int t = 0; t < n_tiles; ++t, ++gt) {
          const int s = gt % STAGES;
          mbar_wait(&S.empty[s], ((gt / STAGES) & 1) ^ 1);
          const int64_t j0 = j_begin + (int64_t)t * BN;
          if constexpr (D == 8) {
            // the D = 8 image is exactly n_rows x 32 B: the last tile is copied short (rows past the table end stay
            // stale: masked in the epilogue)
            const uint32_t wbytes = (uint32_t)min((int64_t)(C::W_FLOATS * 4), (n_rows - j0) * (int64_t)32);
            mbar_expect_tx(&S.full[s], wbytes + C::WT_FLOATS * 4);
            tma_bulk_load(S.w[s], Wsw + j0 * 8, wbytes, &S.full[s]);
          } else {
            // D > 8: the image is zero-padded to whole 256-row tiles of KA atoms [256][32 B]; the BN-row sub-tile of
            // atom a is one contiguous block (its swizzle only depends on row bit 2)
            mbar_expect_tx(&S.full[s], (C::W_FLOATS + C::WT_FLOATS) * 4);
#pragma unroll 1
            for (int a = 0; a < KA; ++a)
              tma_bulk_load(S.w[s] + a * (BN * 8), Wsw + (((j0 >> 8) * KA + a) * (TC_BN * 8) + (j0 & (TC_BN - 1)) * 8),
                            BN * 32, &S.full[s]);
          }
          tma_bulk_load(S.wt[s], Wt + (j0 / BN) * C::WT_FLOATS, C::WT_FLOATS * 4, &S.full[s]);   // zero-padded
        }
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer: scores of tile t, then the gradient MMAs of tile t - 2 (the two epilogue groups work
    // on tiles t - 1 and t - 2 meanwhile; three S/P buffers) ----------------
    {   // all 32 lanes run this block converged (see umma_*_elect)
      uint32_t gt = 0;
      int it = 0;
      auto grad_mma = [&](uint32_t g, bool first_of_item) {   // dq (+)= P(tile g) . Wt(tile g)^T
        const int buf = g % C2_BUFS, s = g % STAGES;
        mbar_wait(&S.pfull[buf], (g / C2_BUFS) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // descriptors of the BN / 8 k-atoms differ only in the start address (NG x 32 B apart): one base, constant offsets
        const uint64_t bd0 = umma_desc_sw32(S.wt[s]);
        const uint32_t pa0 = tmem + buf * BN;
        const uint32_t acc0 = first_of_item ? 0u : 1u;
#pragma unroll
        for (int a = 0; a < BN / 8; ++a)
          umma_tf32_ts_elect(tmem + C::DQ_COL + (a % DQ_ACCS) * NG, pa0 + a * 8, bd0 + (uint64_t)(a * ((NG * 32) >> 4)), IDESC_G,
                             a < DQ_ACCS ? acc0 : 1u);
        umma_commit_elect(&S.tempty[buf]);
        umma_commit_elect(&S.empty[s]);
      };
      for (int w = w_begin; w < w_end; ++w, ++it) {
        const int ab = it % A_BUFS;
        const int n_tiles = item_tiles(w);
        mbar_wait(&S.afull[ab], (it / A_BUFS) & 1);
        if (it > 0) mbar_wait(&S.dqempty, (it - 1) & 1);     // the previous item's gradient has been read out
        const uint64_t adesc = umma_desc_sw32(S.a[ab]);
        for (int t = 0; t < n_tiles; ++t, ++gt) {
          const int buf = gt % C2_BUFS, s = gt % STAGES;
          mbar_wait(&S.tempty[buf], ((gt / C2_BUFS) & 1) ^ 1);
          mbar_wait(&S.full[s], (gt / STAGES) & 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint64_t bdesc = umma_desc_sw32(S.w[s]);
#pragma unroll
          for (int a = 0; a < KA; ++a)   // k-atom a: query atom (4 KB apart) x W atom (BN x 32 B apart)
            umma_tf32_elect(tmem + buf * BN, adesc + (uint64_t)(a * ((TC_BM * 32) >> 4)), bdesc + (uint64_t)(a * ((BN * 32) >> 4)),
                            IDESC_S, a != 0);
          umma_commit_elect(&S.tfull[buf]);
          if (t > 1) grad_mma(gt - 2, t == 2);
        }
        umma_commit_elect(&S.aempty[ab]);          // every score MMA of the item has read the query tile
        if (n_tiles > 1) grad_mma(gt - 2, n_tiles == 2);
        grad_mma(gt - 1, n_tiles == 1);
        umma_commit_elect(&S.dqfull);
      }
    }
  } else {
    // ---------------- epilogue: P = exp(S - c) in place, l += row sums ----------------
    // Two groups of 8 warps ping-pong over the tiles (group g takes the tiles with gt % 2 == g), so one group's TMEM
    // loads / stores / barrier round trips overlap the other group's exponentials.  A warp owns one TMEM lane quarter
    // and one BN/2-column half of its tiles.
    const int quarter = hw_warp & 3;          // TMEM lane quarter = hardware warp id % 4
    const int slice = hw_warp >> 2;           // record stream of this warp (0..3)
    const int group = slice & 1, half = slice >> 1;
    const int trow = quarter * 32 + lane;
    const float LOG2E = 1.4426950408889634f;
    const uint32_t lane_base = tmem + ((uint32_t)(quarter * 32) << 16);
    uint32_t gt = 0;
    int it = 0;
    for (int w = w_begin; w < w_end; ++w, ++it) {
      const int64_t row = item_rows(w) + trow;
      const int64_t j_begin = item_jb(w);
      const int64_t j_end = min(n_rows, j_begin + items_per_split);
      const int n_tiles = item_tiles(w);
      const float nc = (row < M) ? -__ldg(cref + row) * LOG2E : 0.f;
      float l = 0.f;
      int cnt = 0;
      for (int t = 0; t < n_tiles; ++t, ++gt) {
        if ((int)(gt & 1) != group) continue;
        const int buf = gt % C2_BUFS;
        mbar_wait(&S.tfull[buf], (gt / C2_BUFS) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int64_t col0 = j_begin + (int64_t)t * BN + half * HALF;
        const int n_valid = (int)max((int64_t)0, min((int64_t)HALF, j_end - col0));
        cnt += n_valid;
        const uint32_t taddr = lane_base + (uint32_t)(buf * BN + half * HALF);
        uint32_t va[CW], vb[CW];
        c2_ld<CW>(va, taddr);
        if constexpr (NCH == 2) c2_ld<CW>(vb, taddr + CW);
        float l0 = 0.f, l1 = 0.f, l2 = 0.f, l3 = 0.f;
        auto chunk = [&](uint32_t (&v)[CW], int nv) {
          if (nv == CW) {
#pragma unroll
            for (int i = 0; i < CW; i += 4) {
              const float p0 = c2_ex2(fmaf(__uint_as_float(v[i]), LOG2E, nc));
              const float p1 = c2_ex2(fmaf(__uint_as_float(v[i + 1]), LOG2E, nc));
              const float p2 = c2_ex2(fmaf(__uint_as_float(v[i + 2]), LOG2E, nc));
              const float p3 = c2_ex2(fmaf(__uint_as_float(v[i + 3]), LOG2E, nc));
              l0 += p0; l1 += p1; l2 += p2; l3 += p3;
              v[i] = __float_as_uint(p0); v[i + 1] = __float_as_uint(p1);
              v[i + 2] = __float_as_uint(p2); v[i + 3] = __float_as_uint(p3);
            }
          } else {     // last tile of the table: stale scores beyond its end contribute nothing
#pragma unroll
            for (int i = 0; i < CW; ++i) {
              float p0 = c2_ex2(fmaf(__uint_as_float(v[i]), LOG2E, nc));
              if (i >= nv) p0 = 0.f;
              l0 += p0;
              v[i] = __float_as_uint(p0);
            }
          }
        };
        c2_wait_ld<CW>(va);
        chunk(va, min(CW, n_valid));
        c2_st<CW>(taddr, va);
        if constexpr (NCH == 2) {
          c2_wait_ld<CW>(vb);
          chunk(vb, max(0, n_valid - CW));
          c2_st<CW>(taddr + CW, vb);
        }
        l += (l0 + l1) + (l2 + l3);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&S.pfull[buf]);
      }
      float *rec = part + ((int64_t)item_split(w) * M + row) * C::REC;
      // the item's gradient: the slice-0 warps read the DQ_ACCS accumulators (D real columns of NG) once every MMA
      // landed, GW columns at a time, and write their sum into the record's acc[]
      if (slice == 0) {
        mbar_wait(&S.dqfull, it & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
        for (int k0 = 0; k0 < D; k0 += GW) {
          float acc[GW];
#pragma unroll
          for (int k = 0; k < GW; ++k) acc[k] = 0.f;
#pragma unroll
          for (int j = 0; j < DQ_ACCS; ++j) {
            uint32_t g[GW];
            c2_ld<GW>(g, lane_base + (uint32_t)(C::DQ_COL + j * NG + k0));
            c2_wait_ld<GW>(g);
#pragma unroll
            for (int k = 0; k < GW; ++k) acc[k] += __uint_as_float(g[k]);
          }
          if (row < M) {
#pragma unroll
            for (int k = 0; k < GW; ++k) rec[3 + k0 + k] = acc[k];
          }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&S.dqempty);
      }
      // ONE record per (split, row): the other three column slices store their l in shared memory, a named barrier
      // over the four warps of this TMEM lane quarter orders it, the slice-0 warp adds them in slice order (a fixed
      // order: the records, and with them loss and lse, are reproducible bit for bit) and writes the record.  Each
      // buffer is written again two items later, behind the next item's barrier
      float (&ls)[3][TC_BM] = S.lsum[it & 1];
      if (slice != 0) ls[slice - 1][trow] = l;
      asm volatile("bar.sync %0, 128;" ::"r"(1 + quarter) : "memory");
      if (slice == 0) {
        l += (ls[0][trow] + ls[1][trow]) + ls[2][trow];
        if (row < M) {
          rec[0] = __ldg(cref + row);
          rec[1] = l;
          rec[2] = __int_as_float((int)(j_end - j_begin));
        }
      }
      (void)cnt;
    }
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem));
  }
}

// ---------------------------------------------------------------------------
// Table gradient on the tensor cores (pcv_ce_table_grad, engine TF32, dense mask): ce_tc2_kernel with the roles of Q
// and W swapped.  A CTA owns a slab of 128 items (the TMEM lanes) and sweeps every query row, BN at a time:
//
//   S^T[128 items x BN rows] = W_slab . Q_tile^T        KA accumulating tcgen05.mma kind::tf32, A = the slab and B
//                                                       the query tile, both K-major SWIZZLE_32B images in smem
//   P^T = g_i (exp(S^T - lse_i) - [t_i = j])            4 epilogue warps, thread = item: TMEM -> registers -> TMEM
//   dW_slab[128 x NG] += P^T . Qt_tile^T                BN / 8 MMAs, A = P^T from TENSOR MEMORY, B = the transposed
//                                                       query tile [NG dims x BN rows] (the layout of ce_tc2's Wt)
//
// dW stays in TMEM for the whole sweep and is written once: no atomics, no split, reproducible bit for bit.  lse is
// known, so no reference exponent is needed.  The CTA builds its slab and each query tile's two images itself from
// the fp32 arrays (they are small: BN x D floats per image); the steps of a tile run back to back (load, score MMA,
// epilogue, gradient MMA), and the overlap comes from the other CTAs of the SM.
//   D     BN   slab + Q tile + Qt tile (smem)   TMEM columns (S^T + dW, allocated)
//   8    128      4 +  4 +  8 KB                  128 + 16  (256)
//   16   128      8 +  8 +  8 KB                  128 + 16  (256)
//   32   128     16 + 16 + 16 KB                  128 + 32  (256)
//   64    64     32 + 16 + 16 KB                   64 + 64  (128)
//   128   64     64 + 32 + 32 KB                   64 + 128 (256)
// Error: the tf32 logit is within 2^-9 |q_i| |w_j| of the exact one (both operands truncated to 10 mantissa bits), and
// the gradient MMA truncates P^T and Q again (2^-9 relative per term).
template <int D>
struct TgCfg {
  static constexpr int KA = D / 8;
  static constexpr int BN = D <= 32 ? 128 : 64;
  static constexpr int NG = D < 16 ? 16 : D;
  static constexpr int DW_COL = BN;
  static constexpr int TCOLS = (BN + NG) <= 128 ? 128 : 256;
  static constexpr int GW = D < 32 ? D : 32;
};

template <int D>
struct __align__(1024) TgSmem {
  using C = TgCfg<D>;
  float wa[TC_BM * D];             // item slab: KA k-atoms of [128 rows x 32 B]
  float qw[C::BN * D];             // query tile: KA k-atoms of [BN rows x 32 B]
  float qt[(C::BN / 8) * C::NG * 8];   // transposed query tile: BN / 8 k-atoms of [NG rows x 32 B]
  float lse[C::BN], rs[C::BN];
  int64_t tg[C::BN];
  unsigned long long sdone, gdone;
  uint32_t tmem_base;
};

template <int D>
__global__ void __launch_bounds__(TC_BM)
ce_tc_table_grad_kernel(const float *__restrict__ W, int64_t n_rows, const float *__restrict__ Q,
                        const int64_t *__restrict__ targets, const float *__restrict__ lse,
                        const float *__restrict__ row_scale, int64_t M, float *__restrict__ dW) {
  using C = TgCfg<D>;
  constexpr int BN = C::BN, KA = C::KA, NG = C::NG, GW = C::GW;
  constexpr uint32_t IDESC_S = C2_IDESC<BN>, IDESC_G = C2_IDESC<NG>;
  extern __shared__ unsigned char smem_raw[];
  TgSmem<D> &S = *reinterpret_cast<TgSmem<D> *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t j0 = (int64_t)blockIdx.x * TC_BM;

  // item slab, SWIZZLE_32B: row t at byte t*32 of its atom, 16-byte chunk c at ((c ^ bit2(t)) * 16); rows past the
  // table end are zero
  {
    const int64_t j = j0 + tid;
    const int sw = (tid >> 2) & 1;
#pragma unroll
    for (int a = 0; a < KA; ++a) {
      float4 w0 = make_float4(0.f, 0.f, 0.f, 0.f), w1 = w0;
      if (j < n_rows) {
        w0 = __ldg(reinterpret_cast<const float4 *>(W + j * D + a * 8));
        w1 = __ldg(reinterpret_cast<const float4 *>(W + j * D + a * 8) + 1);
      }
      float4 *dst = reinterpret_cast<float4 *>(S.wa + a * (TC_BM * 8) + tid * 8);
      dst[0 ^ sw] = w0;
      dst[1 ^ sw] = w1;
    }
  }
  // the padding rows D..NG-1 of the transposed image stay zero for the whole sweep
  for (int f = tid; f < (BN / 8) * NG * 8; f += TC_BM) S.qt[f] = 0.f;
  if (tid == 0) {
    mbar_init(&S.sdone, 1);
    mbar_init(&S.gdone, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&S.tmem_base)),
                 "r"(C::TCOLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = S.tmem_base;
  const uint32_t lane_base = tmem + ((uint32_t)(warp * 32) << 16);
  const int64_t j = j0 + tid;            // this thread's item = its TMEM lane
  const int n_tiles = (int)((M + BN - 1) / BN);

  for (int t = 0; t < n_tiles; ++t) {
    const int64_t i0 = (int64_t)t * BN;
    // ---- query tile images + its lse / scale / target (rows past M: zero query, zero scale)
    for (int f = tid; f < BN * KA; f += TC_BM) {
      const int r = f / KA, a = f % KA;
      const int64_t i = i0 + r;
      float4 q0 = make_float4(0.f, 0.f, 0.f, 0.f), q1 = q0;
      if (i < M) {
        q0 = __ldg(reinterpret_cast<const float4 *>(Q + i * D + a * 8));
        q1 = __ldg(reinterpret_cast<const float4 *>(Q + i * D + a * 8) + 1);
      }
      const int sw = (r >> 2) & 1;
      float4 *dst = reinterpret_cast<float4 *>(S.qw + a * (BN * 8) + r * 8);
      dst[0 ^ sw] = q0;
      dst[1 ^ sw] = q1;
      // transposed image: element (dim k, row r) of k-atom r / 8 at row k, chunk (r >> 2) & 1 swizzled by bit 2 of k
      const float v[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
      const int ra = r >> 3, c = (r >> 2) & 1, e = r & 3;
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        const int k = a * 8 + kk;
        S.qt[(ra * NG + k) * 8 + ((c ^ ((k >> 2) & 1)) << 2) + e] = v[kk];
      }
    }
    for (int r = tid; r < BN; r += TC_BM) {
      const int64_t i = i0 + r;
      const bool ok = i < M;
      S.lse[r] = ok ? lse[i] : 0.f;
      S.rs[r] = ok ? row_scale[i] : 0.f;
      S.tg[r] = ok ? targets[i] : -1;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // ---- scores S^T = W_slab . Q_tile^T
    if (warp == 0) {
      const uint64_t adesc = umma_desc_sw32(S.wa), bdesc = umma_desc_sw32(S.qw);
#pragma unroll
      for (int a = 0; a < KA; ++a)
        umma_tf32_elect(tmem, adesc + (uint64_t)(a * ((TC_BM * 32) >> 4)), bdesc + (uint64_t)(a * ((BN * 32) >> 4)),
                        IDESC_S, a != 0);
      umma_commit_elect(&S.sdone);
    }
    mbar_wait(&S.sdone, t & 1);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // ---- P^T = g (exp(S^T - lse) - onehot), in place, 32 columns at a time
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      uint32_t v[32];
      TC_LD32(v, lane_base + (uint32_t)c0);
      TC_WAIT_LD(v);
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        const float p = __expf(__uint_as_float(v[c]) - S.lse[c0 + c]);
        v[c] = __float_as_uint(S.rs[c0 + c] * (S.tg[c0 + c] == j ? p - 1.f : p));
      }
      C2_ST32(lane_base + (uint32_t)c0, v);
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // ---- dW_slab += P^T . Qt_tile^T
    if (warp == 0) {
      const uint64_t bd0 = umma_desc_sw32(S.qt);
#pragma unroll
      for (int a = 0; a < BN / 8; ++a)
        umma_tf32_ts_elect(tmem + C::DW_COL, tmem + a * 8, bd0 + (uint64_t)(a * ((NG * 32) >> 4)), IDESC_G,
                           (t == 0 && a == 0) ? 0u : 1u);
      umma_commit_elect(&S.gdone);
    }
    mbar_wait(&S.gdone, t & 1);          // the MMAs have read the tiles and P^T: both may be overwritten
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  }

  // ---- dW rows of this slab, once
#pragma unroll 1
  for (int k0 = 0; k0 < D; k0 += GW) {
    uint32_t g[GW];
    c2_ld<GW>(g, lane_base + (uint32_t)(C::DW_COL + k0));
    c2_wait_ld<GW>(g);
    if (j < n_rows && n_tiles > 0) {
#pragma unroll
      for (int k = 0; k < GW; k += 4)
        *reinterpret_cast<float4 *>(dW + j * D + k0 + k) =
            make_float4(__uint_as_float(g[k]), __uint_as_float(g[k + 1]), __uint_as_float(g[k + 2]), __uint_as_float(g[k + 3]));
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(C::TCOLS));
  }
}

// ------------------------------------------------------------------ host side
struct Ce2Plan {
  int n_split;
  int64_t items_per_split;
  size_t rec_bytes, ws_bytes;   // records; records + cref + flags
};

// The column split is planned in units of 128 items at every D (a multiple of every BN), so a shape gets the same
// split at every dim.
static void ce2_plan(const Table *t, int64_t M, Ce2Plan *p) {
  constexpr int UNIT = 128;
  const int row_tiles = (int)((M + TC_BM - 1) / TC_BM);
  const int64_t tiles = (t->n_rows + UNIT - 1) / UNIT;
  int64_t max_split = tiles / 16;
  if (max_split < 1) max_split = 1;
  if (max_split > 32) max_split = 32;
  int64_t best_ns = 1;
  double best_eff = -1.0;
  for (int64_t ns = 1; ns <= max_split; ++ns) {
    const int64_t tps = (tiles + ns - 1) / ns;
    const int64_t real_ns = (tiles + tps - 1) / tps;
    const int64_t ctas = (int64_t)row_tiles * real_ns;
    const int64_t waves = (ctas + t->sm_count - 1) / t->sm_count;
    const double eff = (double)ctas / (double)(waves * t->sm_count);
    if (eff > best_eff + 0.03) { best_eff = eff; best_ns = real_ns; }
  }
  const int64_t tps = (tiles + best_ns - 1) / best_ns;
  p->n_split = (int)((tiles + tps - 1) / tps);
  p->items_per_split = tps * UNIT;
  const size_t rec = 3 + (size_t)t->dim;
  p->rec_bytes = ((size_t)p->n_split * (size_t)M * rec * sizeof(float) + 255) & ~(size_t)255;   // one record per (split, row)
  p->ws_bytes = p->rec_bytes + (((size_t)M * 4 + 255) & ~(size_t)255) + (((size_t)M + 255) & ~(size_t)255);
}

bool ce_tc_supported(const Table *t) { return tc_dim_ok(t->dim) && t->tmap_valid; }

size_t ce_tc_workspace(const Table *t, int64_t M) {
  if (!ce_tc_supported(t)) return 0;
  Ce2Plan p;
  ce2_plan(t, M, &p);
  return p.ws_bytes;
}

// The transposed image is built on first use (one-off, like the table handle's other packed copy) and owned by it.
// At D >= 16 it is as large as the table itself (D = 8: twice, for the zero rows).
template <int D>
static int ensure_packed_t(Table *t) {
  using C = Ce2Cfg<D>;
  static std::mutex mu;                 // two host threads may hit the first tensor-core CE call of a handle together
  std::lock_guard<std::mutex> lock(mu);
  if (t->packed_t) return PCV_OK;
  const int64_t tiles = (t->n_rows + C::BN - 1) / C::BN;
  const size_t bytes = (size_t)tiles * C::WT_FLOATS * sizeof(float);
  float *p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("ce(tf32): cudaMalloc of the transposed table image (%zu bytes) -> %s", bytes, cudaGetErrorString(e));
    return PCV_ERR_CUDA;
  }
  e = cudaMemset(p, 0, bytes);
  if (e == cudaSuccess) {
    const int64_t n = t->n_rows * D;
    pack_wt_kernel<D><<<(unsigned)((n + 255) / 256), 256>>>(t->W, t->n_rows, p);
    count_launch();
    e = cudaDeviceSynchronize();
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    cudaFree(p);
    set_error("ce(tf32): packing the transposed table image -> %s", cudaGetErrorString(e));
    return PCV_ERR_CUDA;
  }
  t->packed_t = p;
  return PCV_OK;
}

void table_free_ce(Table *t) {
  if (t->packed_t) cudaFree(t->packed_t);
  t->packed_t = nullptr;
}

template <int D>
static int ce_tc_launch_d(Table *t, const Ce2Plan &p, const float *Q, const int64_t *targets, int64_t M, float *part,
                          cudaStream_t st) {
  if (!t->packed_t) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cs);
    if (cs != cudaStreamCaptureStatusNone) {
      set_error("ce(tf32): the first call on a table builds its transposed image and can not run inside a CUDA graph "
                "capture; run one eager step first");
      return PCV_ERR_CUDA;
    }
    const int rc = ensure_packed_t<D>(t);
    if (rc != PCV_OK) return rc;
  }
  float *cref = reinterpret_cast<float *>(reinterpret_cast<char *>(part) + p.rec_bytes);
  unsigned char *unsafe = reinterpret_cast<unsigned char *>(cref) + (((size_t)M * 4 + 255) & ~(size_t)255);
  const int n_streams = p.n_split;
  ce_ref_kernel<D><<<(unsigned)((M + 7) / 8), 256, 0, st>>>(t->W, t->n_rows, t->row_offset, t->max_row_norm_dev(), Q, targets, M,
                                                            cref, unsafe);
  PCV_LAUNCH_CHECK();
  static_assert(sizeof(Ce2Smem<D>) + 1024 <= 227 * 1024, "shared memory of one CTA");
  const size_t smem = sizeof(Ce2Smem<D>) + 1024;
  static bool attr_set[64] = {false};   // one latch per instantiation (a static of this template), per device
  if (!attr_set[t->device & 63]) {
    PCV_CUDA(cudaFuncSetAttribute(ce_tc2_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set[t->device & 63] = true;
  }
  const int64_t n_work = ((M + TC_BM - 1) / TC_BM) * (int64_t)p.n_split;
  const unsigned grid = (unsigned)(n_work < t->sm_count ? n_work : t->sm_count);
  ce_tc2_kernel<D><<<grid, C2_THREADS, smem, st>>>(t->packed, t->packed_t, t->n_rows, Q, M, cref, p.items_per_split,
                                                   p.n_split, (int)n_work, part);
  PCV_LAUNCH_CHECK();
  ce_rowfix_kernel<D><<<(unsigned)((M + 7) / 8), 256, 0, st>>>(t->W, t->n_rows, Q, M, unsafe, n_streams, part);
  PCV_LAUNCH_CHECK();
  return n_streams;
}

// -> number of partial records per row (streams), < 0 on error
int ce_tc_launch(const Table *tc, const float *Q, const int64_t *targets, int64_t M, float *part, size_t ws_bytes, cudaStream_t st) {
  Table *t = const_cast<Table *>(tc);
  Ce2Plan p;
  ce2_plan(t, M, &p);
  if (ws_bytes < p.ws_bytes) {
    set_error("ce(tf32): workspace too small (%zu < %zu)", ws_bytes, p.ws_bytes);
    return PCV_ERR_WORKSPACE;
  }
  switch (t->dim) {
    case 8: return ce_tc_launch_d<8>(t, p, Q, targets, M, part, st);
    case 16: return ce_tc_launch_d<16>(t, p, Q, targets, M, part, st);
    case 32: return ce_tc_launch_d<32>(t, p, Q, targets, M, part, st);
    case 64: return ce_tc_launch_d<64>(t, p, Q, targets, M, part, st);
    case 128: return ce_tc_launch_d<128>(t, p, Q, targets, M, part, st);
  }
  set_error("ce(tf32): dim %d unsupported (use 8, 16, 32, 64 or 128)", t->dim);
  return PCV_ERR_UNSUPPORTED;
}

template <int D>
static int ce_tc_table_grad_d(const Table *t, const float *Q, const int64_t *targets, const float *lse,
                              const float *row_scale, int64_t M, float *dW, cudaStream_t st) {
  static_assert(sizeof(TgSmem<D>) + 1024 <= 227 * 1024, "shared memory of one CTA");
  const size_t smem = sizeof(TgSmem<D>) + 1024;
  static bool attr_set[64] = {false};
  if (!attr_set[t->device & 63]) {
    PCV_CUDA(cudaFuncSetAttribute(ce_tc_table_grad_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set[t->device & 63] = true;
  }
  const unsigned grid = (unsigned)((t->n_rows + TC_BM - 1) / TC_BM);
  ce_tc_table_grad_kernel<D><<<grid, TC_BM, smem, st>>>(t->W, t->n_rows, Q, targets, lse, row_scale, M, dW);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

// tensor-core table gradient (dense mask, dims 8..128): see ce_tc_table_grad_kernel
int ce_tc_table_grad(const Table *t, const float *Q, const int64_t *targets, const float *lse, const float *row_scale,
                     int64_t M, float *dW, cudaStream_t st) {
  switch (t->dim) {
    case 8: return ce_tc_table_grad_d<8>(t, Q, targets, lse, row_scale, M, dW, st);
    case 16: return ce_tc_table_grad_d<16>(t, Q, targets, lse, row_scale, M, dW, st);
    case 32: return ce_tc_table_grad_d<32>(t, Q, targets, lse, row_scale, M, dW, st);
    case 64: return ce_tc_table_grad_d<64>(t, Q, targets, lse, row_scale, M, dW, st);
    case 128: return ce_tc_table_grad_d<128>(t, Q, targets, lse, row_scale, M, dW, st);
  }
  set_error("ce_table_grad(tf32): dim %d unsupported (use 8, 16, 32, 64 or 128)", t->dim);
  return PCV_ERR_UNSUPPORTED;
}

}  // namespace pcv
