// score_select_tc.cu — greedy score+select on the 5th-gen tensor cores (sm_100a).
//
// Same contract as score_select.cu (cvae.py:97-101, pivotcvae.py:191): bit-exact
// arg-max of the fp32 sequential-k FMA chain, ties -> lowest index.  The tensor
// cores only FILTER:
//
//   1. The table handle keeps a PRE-SWIZZLED copy of the frozen table (rows with bit 2
//      of the row index set have their two 16-byte halves swapped = the K-major
//      SWIZZLE_32B shared-memory image).  One TMA bulk copy (cp.async.bulk, 8 KB,
//      a single contiguous request) per 256-item tile streams it into a 12-stage
//      shared-memory ring.  (A 2-D tensor-map load with a 32-byte inner box was
//      measured ~8x slower: one 32 B request per row; see profiles/.)
//   2. One elected thread issues tcgen05.mma.kind::tf32, M=128 (query rows, staged
//      once per CTA), N=256, K=8 per tile; accumulators ping-pong between two
//      256-column TMEM buffers (512 columns = all of TMEM).
//   3. SEL_EPI_WARPS epilogue warps read their TMEM lanes (tcgen05.ld 32x32b.x32: thread =
//      query row), keep a running max r of the APPROXIMATE scores and record every
//      32-item chunk whose approximate maximum is >= r - band in a per-row
//      shared-memory list (fast path: 16 FMNMX3 + 1 compare per 32 logits).
//      band = 2*eps, eps = 1.25 * 2^-9 * |q|_2 * max_j |w_j|_2 bounds |tf32 - fp32 chain|
//      (both operands truncated to 10 mantissa bits: relative 2^-10 each), so the
//      exact arg-max (and every exact tie) is always in the list.
//   4. Each (row, CTA slot, column-slice) stream hands its running max and its (<= 4)
//      surviving chunks to tc_refine_kernel: one warp per row takes R = max over the
//      streams, and re-scores item-by-item (lane = item, coalesced 1 KB reads) every
//      chunk still inside the band of R with the exact fp32 FMA chain from the fp32
//      table; winner = largest exact score, ties -> lowest index.
//   5. Chunks that do not fit a stream's lists (heavy exact ties) spill to the CTA's region
//      of an overflow list and are re-scored exactly at the end of the filter kernel itself
//      (packed 64-bit atomicMax per row, folded in by the refine kernel).
//
// The (M x N) logits never leave TMEM, and the result is exact for any input
// (streams whose overflow region is full too are flagged and scanned exactly by the
// refine kernel).
#include <cstdlib>
#include <cuda_fp16.h>

#include "table_images.cuh"

namespace pcv {

// Optional phase trace of CTA 0 (profiles/trace_select.py builds a separate library with -DPCV_TC_TRACE).
#ifdef PCV_TC_TRACE
__device__ long long g_tc_trace[16];
__device__ long long g_tc_mma[16];   // MMA issuer, tiles 40..43: tempty passed / operands ready (just before the issue)
__device__ long long g_tc_cta[4][256];   // per CTA: clock64 at entry / exit, globaltimer at entry / exit
__device__ __forceinline__ long long tc_gtime() { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define TC_TRACE(i) do { if (blockIdx.x == 0) g_tc_trace[i] = clock64();                                          \
    if ((i) == 0) { g_tc_cta[0][blockIdx.x & 255] = clock64(); g_tc_cta[2][blockIdx.x & 255] = tc_gtime(); }      \
    if ((i) == 14) { g_tc_cta[1][blockIdx.x & 255] = clock64(); g_tc_cta[3][blockIdx.x & 255] = tc_gtime(); } } while (0)
#else
#define TC_TRACE(i) do { } while (0)
#endif

// The epilogue is latency-bound per warp (TMEM load -> max tree -> compare -> branch), so it runs
// 16 warps: four per TMEM lane quarter, each owning a 64-column slice of every 256-column tile.
constexpr int SEL_EPI_WARPS = 16;                     // multiple of 4 (a warp reads one TMEM lane quarter)
constexpr int SEL_SLICES = SEL_EPI_WARPS / 4;         // column slices of a tile
constexpr int SEL_SW = TC_BN / SEL_SLICES;            // columns per slice
constexpr int SEL_THREADS = 64 + 32 * SEL_EPI_WARPS;  // warp 0 TMA, warp 1 MMA/TMEM, then the epilogue warps
constexpr int TC_OUT = 4;                            // recorded chunks handed to the refine kernel per (stream, row)

// The embedding dimension D = 8 * KA is walked in K-ATOMS of 8 fp32 (= 32 bytes = one kind::tf32 k-step).  Operand
// tiles are stored k-atom-major, each atom a [rows][32 B] SWIZZLE_32B image, so the D = 8 layout (KA = 1) is
// the special case and a larger D only adds MMAs (accumulating in TMEM) per table tile, not a new layout:
//   table tile j: packed[(j * KA + a) * 2048 floats ..]  = atom a of rows 256 j .. 256 j + 255
//   ring stage  : KS consecutive atoms of one tile (one TMA bulk copy of KS * 8 KB)
template <int KA>
struct TcCfg {
  static constexpr int D = 8 * KA;
  static constexpr int KS = KA == 1 ? 1 : 2;          // k-atoms per ring stage
  static constexpr int STAGES = KA == 1 ? 12 : 6;     // 96 KB of table tiles in flight
  static constexpr int A_BUFS = KA <= 8 ? 2 : 1;      // query tiles: double-buffered across segments while they fit
  static constexpr int CAP = KA <= 4 ? 16 : 8;        // in-kernel recorded-chunk list capacity per (slice, row)
  static constexpr int ATOM_A = TC_BM * 8;            // floats per k-atom of the query tile
  static constexpr int ATOM_B = TC_BN * 8;            // floats per k-atom of a table tile
  static constexpr uint32_t STAGE_BYTES = KS * ATOM_B * 4;
};

template <int KA>
struct __align__(1024) TcSmem {
  using C = TcCfg<KA>;
  float b[C::STAGES][C::KS * C::ATOM_B];       // SWIZZLE_32B tile atoms written by TMA
  float a[C::A_BUFS][KA * C::ATOM_A];          // query tiles, same layout
  unsigned long long cand[SEL_SLICES][C::CAP][TC_BM];  // recorded 32-item chunks per (slice, row): (approx max bits << 32) | first item
  float rmax[TC_BM];                           // running max per row, shared by the column slices
  unsigned long long full[C::STAGES], empty[C::STAGES], tfull[2], tempty[2], afull[2], aempty[2];
  uint32_t tmem_base;
  unsigned int ovf_n;                           // overflow entries this CTA has spilled to its region of the global list
};

// exact fp32 sequential-k FMA chain (SURVEY F3) of one item against a query row held in global memory
template <int D>
__device__ __forceinline__ float tc_exact_score(const float *__restrict__ q, const float *__restrict__ w) {
  float sc = 0.f;
#pragma unroll
  for (int k = 0; k < D; k += 4) {
    const float4 q4 = __ldg(reinterpret_cast<const float4 *>(q + k));
    const float4 w4 = __ldg(reinterpret_cast<const float4 *>(w + k));
    sc = fmaf(q4.x, w4.x, sc); sc = fmaf(q4.y, w4.y, sc); sc = fmaf(q4.z, w4.z, sc); sc = fmaf(q4.w, w4.w, sc);
  }
  return sc;
}
// |q|^2 with the same left-to-right FMA chain everywhere it is needed (filter and refine must agree on the band)
template <int D>
__device__ __forceinline__ float tc_norm2(const float *__restrict__ q) {
  float ss = 0.f;
#pragma unroll
  for (int k = 0; k < D; k += 4) {
    const float4 q4 = __ldg(reinterpret_cast<const float4 *>(q + k));
    ss = fmaf(q4.x, q4.x, ss); ss = fmaf(q4.y, q4.y, ss); ss = fmaf(q4.z, q4.z, ss); ss = fmaf(q4.w, q4.w, ss);
  }
  return ss;
}

// |q| for the tf32 filter's band, from ss = tc_norm2.  Where |q|^2 under- or overflows (|q| outside ~[1e-15, 1e15])
// the chain is re-summed on q scaled by 2^+-64, which is exact, so that the band still follows |q|: a band collapsed
// to 1e-37 would let the refine drop the chunk of the true arg-max of a tiny row.  Filter and refine both call this.
template <int D>
__device__ __noinline__ float tc_norm_rescaled(const float *__restrict__ q, float s) {
  float ss = 0.f;
#pragma unroll
  for (int k = 0; k < D; ++k) {
    const float v = __ldg(q + k) * s;
    ss = fmaf(v, v, ss);
  }
  return sqrtf(ss) / s;
}
template <int D>
__device__ __forceinline__ float tc_norm(const float *__restrict__ q, float ss) {
  return (ss >= 0x1p-100f && ss <= 0x1p100f) ? sqrtf(ss) : tc_norm_rescaled<D>(q, ss < 1.f ? 0x1p64f : 0x1p-64f);
}

// max of 32 accumulator values; g[0..10] are the maxima of the 3-element groups
// (g[10] covers elements 30, 31) so the rare slow path can skip whole groups.
__device__ __forceinline__ float chunk_max(const uint32_t (&v)[32], float (&g)[11]) {
#pragma unroll
  for (int i = 0; i < 10; ++i)
    g[i] = max3(__uint_as_float(v[3 * i]), __uint_as_float(v[3 * i + 1]), __uint_as_float(v[3 * i + 2]));
  g[10] = fmaxf(__uint_as_float(v[30]), __uint_as_float(v[31]));
  float a = max3(g[0], g[1], g[2]), b = max3(g[3], g[4], g[5]), c = max3(g[6], g[7], g[8]);
  return max3(max3(a, b, c), g[9], g[10]);
}

// ---- f16 filter (D = 8): kind::f16 MMA with f16 accumulators.  An f16 accumulator occupies one 32-bit TMEM column
// (low half), but tcgen05.ld ... .pack::16b returns two columns per register at twice the fp32 element rate
// (profiles/micro/tmem_f16.cu: 142 vs 277 cycles per 128 x 256 tile), and VIMNMX3.U16x2 takes the maximum of SIX
// 16-bit values per instruction — IF the approximate scores are non-negative, so that their f16 bit patterns order
// like unsigned integers.  kind::f16 has K = 16 and D = 8 uses half of it: dimension 8 carries a constant,
// q'_8 = w_8 = 1, and the query row is scaled so that |q'| max|w| = 0.987:
//     a~ = sum_k f16(q'_k) f16(w_k) + 1   in (0, 2),   |a~ - (s' + 1)| <= 2^-10 (operands, RN) + 2^-10 (result) = 2^-9.
// Scaling a row by 2^-e does not move its arg-max, so the filter runs entirely in that scaled, shifted domain with the
// CONSTANT band 2 * 1.25 * 2^-9; the refine re-scores the surviving chunks with the exact fp32 chain as before.
// (The scale is 0.99 / (|q| max|w| 1.003), not a power of two: see tc_h_scale.)  Rows the scale cannot serve get q' = 0
// instead: every approximate score is then the constant 1, their streams overflow and are scanned exactly.
constexpr float TC_H_BAND = 2.0f * 1.25f * 0.001953125f;
constexpr uint32_t TC_IDESC_F16 = (0u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(TC_BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);

__device__ __forceinline__ void umma_f16_elect(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p, q;\n"
      "elect.sync _|q, 0xffffffff;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// 64 TMEM columns of f16 accumulators -> 32 registers of two (column 2i in the low half, 2i + 1 in the high half)
#define TC_LD32_PACK16(v, taddr)                                                                            \
  asm volatile(                                                                                             \
      "tcgen05.ld.sync.aligned.32x32b.x32.pack::16b.b32 "                                                   \
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "                             \
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"             \
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),     \
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),            \
        "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]),          \
        "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]),          \
        "=r"(v[29]), "=r"(v[30]), "=r"(v[31])                                                               \
      : "r"(taddr))
// packed unsigned maximum of 16 registers (32 values): 7 VIMNMX3.U16x2 -> two registers whose maximum is the chunk's
__device__ __forceinline__ void chunk_max_u16x2(const uint32_t *v, uint32_t &b0, uint32_t &b1) {
  const uint32_t a0 = __vimax3_u16x2(v[0], v[1], v[2]), a1 = __vimax3_u16x2(v[3], v[4], v[5]);
  const uint32_t a2 = __vimax3_u16x2(v[6], v[7], v[8]), a3 = __vimax3_u16x2(v[9], v[10], v[11]);
  const uint32_t a4 = __vimax3_u16x2(v[12], v[13], v[14]);
  b0 = __vimax3_u16x2(a0, a1, a2);
  b1 = __vimax3_u16x2(a3, a4, v[15]);
}
// scale of a query row of the f16 filter: |q'| max|w| = 0.99 / 1.003 (wmax_s is max|w| inflated by 0.3 %).  The scale
// need not be a power of two: q' = fl(c q) adds 2^-24 relative to an error budget of 2^-10, and a positive scale does
// not move the row's arg-max.  Keeping the product at the TOP of [0.5, 1) matters: the band is a constant of the scaled
// domain, so relative to |q| it is 1 / (|q'| max|w|) times wider — at 0.5 twice the tf32 filter's, and with it the
// number of chunks a stream hands over (measured at 10 M items: streams overflowing their four hand-over slots and
// being re-scanned exactly made the refine 200x slower).
// ss below 2^-100 (|q| < ~1e-15) may be a subnormal that has lost most of its bits: a scale from it could put
// |q'| max|w| above 1 and a~ below 0, whose f16 sign bit wins the unsigned maxima.  Such rows get q' = 0 as well.
__device__ __forceinline__ float tc_h_scale(float ss, float wmax_s) {
  const float t = sqrtf(ss) * wmax_s;
  if (!(ss >= 0x1p-100f) || !(t > 1.0e-30f) || !(t < 1.0e30f)) return 0.f;   // zero, tiny, huge or non-finite row: q' = 0
  return 0.99f / t;
}

// Packed exact winner of a row among its overflow chunks, merged with a 64-bit atomicMax:
// (order-preserving float bits << 32) | (0xffffffff - item) -> largest score, then lowest index.
__device__ __forceinline__ unsigned long long pack_best(float v, int32_t j) {
  v = v + 0.0f;  // -0 -> +0 so that equal scores compare equal
  uint32_t b = __float_as_uint(v);
  b = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  return ((unsigned long long)b << 32) | (uint32_t)(0xffffffffu - (uint32_t)j);
}
__device__ __forceinline__ void unpack_best(unsigned long long p, float *v, int32_t *j) {
  uint32_t b = (uint32_t)(p >> 32);
  b = (b & 0x80000000u) ? (b & 0x7fffffffu) : ~b;
  *v = __uint_as_float(b);
  *j = (int32_t)(0xffffffffu - (uint32_t)p);
}

// Append one chunk to this CTA's region of the overflow list; true when the region is full.  Out of line on
// purpose: inlined, its address arithmetic gets hoisted into the per-chunk fast path.
__device__ __noinline__ bool tc_spill(unsigned int *ovf_n, unsigned long long *__restrict__ ovf_ent,
                                      int32_t *__restrict__ ovf_row, unsigned int cap, unsigned long long ent, int32_t row) {
  const unsigned int pos = atomicAdd(ovf_n, 1u);
  if (pos >= cap) return true;
  const size_t o = (size_t)blockIdx.x * cap + pos;
  ovf_ent[o] = ent;
  ovf_row[o] = row;
  return false;
}

// One warp per spilled chunk (lane = item): exact fp32 re-score, the winner is merged into row_best[row],
// which tc_refine_kernel folds into the row's result.
template <int D>
__device__ __noinline__ void tc_rescore_overflow(const float *__restrict__ W, int64_t n_rows, const float *__restrict__ Q,
                                                 const unsigned long long *__restrict__ ent, const int32_t *__restrict__ rows,
                                                 unsigned int n, unsigned long long *__restrict__ row_best) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (unsigned int i = warp; i < n; i += blockDim.x >> 5) {
    const int64_t row = rows[i];
    const int64_t j = (int64_t)(uint32_t)ent[i] + lane;
    float best = -INFINITY;
    int32_t bidx = 0x7fffffff;
    if (j < n_rows) {
      best = tc_exact_score<D>(Q + row * D, W + j * D);
      bidx = (int32_t)j;
    }
    if (!(best > -INFINITY)) { best = -INFINITY; bidx = 0x7fffffff; }   // a NaN never wins (nor poisons the merge)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, best, o);
      const int32_t oi = __shfl_xor_sync(0xffffffffu, bidx, o);
      if (ov > best || (ov == best && oi < bidx)) { best = ov; bidx = oi; }
    }
    if (lane == 0 && bidx != 0x7fffffff) atomicMax(row_best + row, pack_best(best, bidx));
  }
}

// Work decomposition: the (row tile, table tile) pairs form one flat sequence of n_units =
// row_tiles * T units (T = table tiles per row tile); CTA c of G owns the contiguous units
// [c*n_units/G, (c+1)*n_units/G) and cuts them at row-tile boundaries into SEGMENTS
// (row tile, [ct0, ct1)).  A row tile is therefore touched by a handful of consecutive CTAs
// (<= ceil(T / (n_units/G)) + 1): its "slots", numbered from the first CTA that touches it.
__host__ __device__ __forceinline__ int64_t tc_cta_begin(int64_t c, int64_t n_units, int G) { return c * n_units / G; }
// the CTA that owns unit x: the largest c with tc_cta_begin(c) <= x
__host__ __device__ __forceinline__ int tc_cta_of(int64_t x, int64_t n_units, int G) {
  return (int)(((x + 1) * G - 1) / n_units);
}

// PERSISTENT: one CTA per SM walks its segments; TMEM, the mbarrier rings and the TMA pipeline
// live across segments, so the per-segment cost is just the tile stream.  Roles:
//   warp 0  : stages the NEXT item's 128 query rows into the double-buffered A tile (all lanes),
//             then lane 0 streams that item's table tiles with TMA bulk copies;
//   warp 1  : lane 0 issues one tcgen05.mma per tile (TMEM alloc/dealloc by the whole warp);
//   warps 2+: epilogue (thread = query row x column slice).
template <int KA, bool F16 = false>
__global__ void __launch_bounds__(SEL_THREADS, 1)
score_select_tc_kernel(const float *__restrict__ Wsw, const float *__restrict__ W, int64_t n_rows,
                       const float *__restrict__ Q, int64_t M, int T, int Tc, int row_tiles, int slots_max,
                       const float *__restrict__ max_row_norm /* the handle's device scalar */, float *__restrict__ out_r, int32_t *__restrict__ out_cnt,
                       unsigned long long *__restrict__ out_ent, unsigned long long *__restrict__ row_best,
                       unsigned long long *__restrict__ ovf_ent, int32_t *__restrict__ ovf_row, unsigned int ovf_cta_cap) {
  using C = TcCfg<KA>;
  constexpr int D = C::D;
  static_assert(!F16 || KA == 1, "the f16 filter is built for D = 8");
  extern __shared__ unsigned char smem_raw[];
  TcSmem<KA> &S = *reinterpret_cast<TcSmem<KA> *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) TC_TRACE(0);
  const float wmax = __ldg(max_row_norm);
  const float band_scale = tc_band_scale(F16, wmax);   // F16: max|w| * 1.003
  // f16 filter on a table refreshed out of the f16 range: every stream is flagged, the refine scans them exactly
  const bool flag_all = F16 && !tc_f16_in_range(wmax);

  if (threadIdx.x == 0) {
    S.ovf_n = 0u;
    for (int s = 0; s < C::STAGES; ++s) { mbar_init(&S.full[s], 1); mbar_init(&S.empty[s], 1); }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&S.tfull[b], 1); mbar_init(&S.tempty[b], SEL_EPI_WARPS);
      mbar_init(&S.afull[b], 1); mbar_init(&S.aempty[b], 1);
    }
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
  if (threadIdx.x == 0) TC_TRACE(1);

  // COLUMN CHUNKS: a catalog that does not fit the L2 is walked chunk by chunk (Tc tiles = 32 MB each); inside a
  // chunk the (row tile, table tile) units are cut evenly over the CTAs as before.  All CTAs are therefore in the
  // same chunk at (about) the same time and share its tiles through the L2 instead of each streaming the whole
  // table from HBM (C5, 10 M items: 1.9 T -> ~13 T logits/s).  T <= Tc: one chunk, the original partition.
  const int n_chunks = (T + Tc - 1) / Tc;
#define TC_CHUNK(ch)                                                                                   \
  const int Tch = min(Tc, T - (ch) * Tc);                                                              \
  const int64_t n_units = (int64_t)row_tiles * Tch;                                                    \
  const int64_t u_begin = tc_cta_begin(blockIdx.x, n_units, gridDim.x);                                \
  const int64_t u_end = tc_cta_begin(blockIdx.x + 1, n_units, gridDim.x);                              \
  const int tile0 = (ch) * Tc; /* first table tile of the chunk */
  // segment starting at unit u: row tile rt, table tiles tile0 + [ct0, ct0 + n_tiles)
#define TC_SEGMENT(u)                                                            \
  const int rt = (int)((u) / Tch);                                               \
  const int ct0 = (int)((u) - (int64_t)rt * Tch);                                \
  const int n_tiles = (int)min((int64_t)(Tch - ct0), u_end - (u));               \
  const int64_t j_begin = (int64_t)(tile0 + ct0) * TC_BN;                        \
  const int64_t j_end = min(n_rows, (int64_t)(tile0 + ct0 + n_tiles) * TC_BN);

  if (warp == 0) {
    // ---------------- producer: A tile of the item, then its table tiles ----------------
    uint32_t gs = 0;   // ring stages issued so far (KA / KS per table tile)
    int it = 0;        // items started so far
    for (int ch = 0; ch < n_chunks; ++ch) {
    TC_CHUNK(ch)
    for (int64_t u = u_begin; u < u_end; ++it) {
      TC_SEGMENT(u)
      u += n_tiles;
      (void)j_end;
      const int ab = it % C::A_BUFS;
      mbar_wait(&S.aempty[ab], ((it / C::A_BUFS) & 1) ^ 1);   // MMAs of the segment that used this A buffer are done
      {
        // 128 query rows per k-atom: row t at byte t*32, 16-byte chunk c at ((c ^ bit2(t)) * 16)  (SWIZZLE_32B image)
        const int64_t row_base = (int64_t)rt * TC_BM;
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
            if constexpr (F16) {
              // 16 f16 per row: the 8 scaled dimensions, then the constant dimension (1 for live rows) and zeros
              float ss = 0.f;
              ss = fmaf(q0.x, q0.x, ss); ss = fmaf(q0.y, q0.y, ss); ss = fmaf(q0.z, q0.z, ss); ss = fmaf(q0.w, q0.w, ss);
              ss = fmaf(q1.x, q1.x, ss); ss = fmaf(q1.y, q1.y, ss); ss = fmaf(q1.z, q1.z, ss); ss = fmaf(q1.w, q1.w, ss);
              const float sc = tc_h_scale(ss, band_scale);
              if (sc == 0.f) { q0 = make_float4(0.f, 0.f, 0.f, 0.f); q1 = q0; }   // (inf * 0 would be NaN)
              const __half2 h0 = __floats2half2_rn(q0.x * sc, q0.y * sc), h1 = __floats2half2_rn(q0.z * sc, q0.w * sc);
              const __half2 h2 = __floats2half2_rn(q1.x * sc, q1.y * sc), h3 = __floats2half2_rn(q1.z * sc, q1.w * sc);
              q0 = make_float4(__uint_as_float(*reinterpret_cast<const uint32_t *>(&h0)), __uint_as_float(*reinterpret_cast<const uint32_t *>(&h1)),
                               __uint_as_float(*reinterpret_cast<const uint32_t *>(&h2)), __uint_as_float(*reinterpret_cast<const uint32_t *>(&h3)));
              q1 = make_float4(__uint_as_float(row < M ? 0x00003C00u : 0u), 0.f, 0.f, 0.f);
            }
            float4 *dst = reinterpret_cast<float4 *>(S.a[ab] + a * C::ATOM_A + t * 8);
            dst[0 ^ sw] = q0;
            dst[1 ^ sw] = q1;
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&S.afull[ab]);
        if (lane == 0 && it == 0) TC_TRACE(2);
      }
      if (lane == 0) {
        for (int t = 0; t < n_tiles; ++t) {
          const int64_t j0 = j_begin + (int64_t)t * TC_BN;
#pragma unroll 1
          for (int kg = 0; kg < KA / C::KS; ++kg, ++gs) {
            const int s = gs % C::STAGES;
            const uint32_t ph = (gs / C::STAGES) & 1;
            mbar_wait(&S.empty[s], ph ^ 1);
            // D = 8: the packed copy is exactly n_rows x 32 B, the last tile is short (rows past the end of the
            // table keep stale data: masked in the epilogue); D > 8: the copy is padded to whole tiles
            const uint32_t bytes = KA == 1 ? (uint32_t)min((int64_t)C::STAGE_BYTES, (n_rows - j0) * (int64_t)32) : C::STAGE_BYTES;
            mbar_expect_tx(&S.full[s], bytes);
            tma_bulk_load(S.b[s], Wsw + j0 * D + (int64_t)kg * (C::KS * C::ATOM_B), bytes, &S.full[s]);
            if (gs == 0) TC_TRACE(3);
          }
        }
      }
      __syncwarp();
    }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer (the whole warp, converged; one elected lane issues: tc_common.cuh) ----------------
    {
      uint32_t gt = 0, gs = 0;
      int it = 0;
      for (int ch = 0; ch < n_chunks; ++ch) {
      TC_CHUNK(ch)
      for (int64_t u = u_begin; u < u_end; ++it) {
        TC_SEGMENT(u)
        u += n_tiles;
        (void)j_begin; (void)j_end;
        const int ab = it % C::A_BUFS;
        mbar_wait(&S.afull[ab], (it / C::A_BUFS) & 1);
        const uint64_t adesc = umma_desc_sw32(S.a[ab]);
        for (int t = 0; t < n_tiles; ++t, ++gt) {
          const int buf = gt & 1;
          const uint32_t bph = (gt >> 1) & 1;
          mbar_wait(&S.tempty[buf], bph ^ 1);
#ifdef PCV_TC_TRACE
          if (blockIdx.x == 0 && gt >= 40 && gt < 44) g_tc_mma[2 * (gt - 40)] = clock64();
#endif
#pragma unroll 1
          for (int kg = 0; kg < KA / C::KS; ++kg, ++gs) {
            const int s = gs % C::STAGES;
            const uint32_t ph = (gs / C::STAGES) & 1;
            mbar_wait(&S.full[s], ph);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#ifdef PCV_TC_TRACE
            if (blockIdx.x == 0 && gt >= 40 && gt < 44) g_tc_mma[2 * (gt - 40) + 1] = clock64();
#endif
            if (gt == 0) TC_TRACE(4);
            // one k-step (8 fp32 = 32 B) per k-atom: the descriptors step by whole atoms (4 KB of A, 8 KB of B)
#pragma unroll
            for (int a = 0; a < C::KS; ++a) {
              if constexpr (F16)
                umma_f16_elect(tmem + buf * TC_BN, adesc, umma_desc_sw32(S.b[s]), TC_IDESC_F16, 0);
              else
                umma_tf32_elect(tmem + buf * TC_BN, adesc + (uint64_t)(((kg * C::KS + a) * C::ATOM_A * 4) >> 4),
                                umma_desc_sw32(S.b[s] + a * C::ATOM_B), TC_IDESC, (kg | a) != 0);
            }
            umma_commit_elect(&S.empty[s]);
          }
          umma_commit_elect(&S.tfull[buf]);
        }
        umma_commit_elect(&S.aempty[ab]);   // fires when every MMA of this item has read the A tile
      }
      }
    }
  } else {
    // ---------------- epilogue: thread = (query row, column slice) ----------------
    const int quarter = warp & 3;             // TMEM lane quarter this warp may read
    const int slice = (warp - 2) >> 2;        // which SEL_SW columns of every 256-column tile
    const int trow = quarter * 32 + lane;
    unsigned long long *list = &S.cand[slice][0][trow];  // entry e at list[e * TC_BM]
    // loop invariants pinned in registers (an opaque mov keeps the compiler from re-deriving them per tile)
    uint32_t tfull_u32, tempty_u32, taddr0;
    asm volatile("mov.u32 %0, %1;" : "=r"(tfull_u32) : "r"(smem_u32(&S.tfull[0])));
    asm volatile("mov.u32 %0, %1;" : "=r"(tempty_u32) : "r"(smem_u32(&S.tempty[0])));
    asm volatile("mov.u32 %0, %1;" : "=r"(taddr0) : "r"(tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(slice * SEL_SW)));
    uint32_t gt = 0;
    float r = 0.f, thr = 0.f, band = 0.f;   // per-row state of the current segment
    uint32_t thrm2 = 0u;                    // F16: (f16 bits of thr rounded down) - 1 in both halves: a chunk passes iff some value > it
    auto pack_thr = [&]() {
      if constexpr (F16) {
        uint32_t t16 = 0u;
        if (thr > 0.f) t16 = (uint32_t)__half_as_ushort(__float2half_rd(thr));   // +inf (dummy rows) -> 0x7C00: nothing passes
        const uint32_t tm = t16 ? t16 - 1u : 0u;
        thrm2 = tm * 0x10001u;
      }
    };
    for (int ch = 0; ch < n_chunks; ++ch) {
    TC_CHUNK(ch)
    for (int64_t u = u_begin; u < u_end;) {
      TC_SEGMENT(u)
      u += n_tiles;
      const int64_t row = (int64_t)rt * TC_BM + trow;
      const bool live = row < M;
      {   // every segment starts on new rows: reset the running max
        if constexpr (F16) {
          band = TC_H_BAND;     // constant in the scaled, shifted domain of the approximate scores
        } else {
          float nq = 0.f;
          if (live) nq = tc_norm<D>(Q + row * D, tc_norm2<D>(Q + row * D));
          band = band_scale * nq * 1.0001f + 1e-37f;
        }
        // running max of the approximate scores; finite start so that masked (-inf) columns
        // never pass, +inf for dummy rows so that nothing ever passes
        r = live ? -3.0e38f : INFINITY;
        thr = r;
        pack_thr();
        atomicExch(reinterpret_cast<unsigned int *>(&S.rmax[trow]), __float_as_uint(-3.0e38f));   // shared with the other column slices
      }
      int cnt = 0;
      bool ovf = false;
      // rare: more chunks inside the band than a list holds -> append them to this CTA's region of the
      // overflow list (re-scored exactly at the end of the kernel); only if that is full too is the stream flagged
      auto spill = [&](unsigned long long ent) {
        if (tc_spill(&S.ovf_n, ovf_ent, ovf_row, ovf_cta_cap, ent, (int32_t)row)) ovf = true;
      };
      // a full list is compacted in place: chunks whose approximate maximum fell out of the
      // band of the (grown) running max can never hold the winner
      auto compact = [&]() {
        int k = 0;
        for (int e = 0; e < cnt; ++e) {
          const unsigned long long ent = list[e * TC_BM];
          if (__uint_as_float((uint32_t)(ent >> 32)) >= thr) list[(k++) * TC_BM] = ent;
        }
        cnt = k;
      };
      // one 32-column chunk: 16 FMNMX3 + one compare; a chunk whose approximate maximum is
      // inside the band of the running max is only RECORDED (one shared-memory store) — the
      // exact fp32 re-score happens in the refine kernel
      auto process = [&](uint32_t (&v)[32], int32_t jb) {
        float g[11];
        const float m = chunk_max(v, g);
        if (m >= thr) {
          r = fmaxf(r, m);
          thr = r - band;
          if (cnt == C::CAP) compact();
          if (cnt < C::CAP) {
            list[cnt * TC_BM] = ((unsigned long long)__float_as_uint(m) << 32) | (uint32_t)jb;
            ++cnt;
          } else {
            spill(((unsigned long long)__float_as_uint(m) << 32) | (uint32_t)jb);
          }
        }
      };
      // f16 filter: 32 items = 16 packed registers; 7 VIMNMX3.U16x2 + one against the packed threshold
      auto process_h = [&](const uint32_t *v, int32_t jb) {
        uint32_t b0, b1;
        chunk_max_u16x2(v, b0, b1);
        if (__vimax3_u16x2(b0, b1, thrm2) != thrm2) {     // some approximate score >= f16(thr)
          const uint32_t bm = __vmaxu2(b0, b1);
          const uint32_t m16 = max(bm & 0xffffu, bm >> 16);
          const float m = __half2float(__ushort_as_half((unsigned short)m16));
          r = fmaxf(r, m);
          thr = r - band;
          pack_thr();
          if (cnt == C::CAP) compact();
          if (cnt < C::CAP) {
            list[cnt * TC_BM] = ((unsigned long long)__float_as_uint(m) << 32) | (uint32_t)jb;
            ++cnt;
          } else {
            spill(((unsigned long long)__float_as_uint(m) << 32) | (uint32_t)jb);
          }
        }
      };
      auto mask_tail = [&](uint32_t (&v)[32], int col0, int n_valid) {
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (col0 + i >= n_valid) v[i] = 0xff800000u;  // -inf: stale / foreign columns never win
      };

      constexpr int NCH = SEL_SW / 32;  // chunks per slice per tile (even)
      // per-tile bookkeeping kept to 32-bit adds: shared addresses of the barriers, the first item of this
      // slice in the tile, the number of tiles that need no tail mask
      const int n_full = max(0, min(n_tiles, (int)(n_rows / TC_BN) - (tile0 + ct0)));
      const bool exch = live && n_tiles >= 8;
      int32_t jb0 = (int32_t)j_begin + slice * SEL_SW;
      for (int t = 0; t < n_tiles; ++t, ++gt, jb0 += TC_BN) {
        const uint32_t buf = gt & 1;
        mbar_wait_u32(tfull_u32 + buf * 8, (gt >> 1) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (threadIdx.x == 64 && gt >= 40 && gt < 44) TC_TRACE(5 + 2 * (gt - 40));
        const uint32_t taddr = taddr0 + buf * TC_BN;
        bool released = false;     // the TMEM buffer goes back as soon as this warp's columns are in registers
        uint32_t va[32], vb[32];
        // software pipeline: the TMEM load of chunk c+1 is in flight while chunk c is reduced
        // (f16 filter: ONE packed load brings the slice's 64 columns)
        if constexpr (F16) TC_LD32_PACK16(va, taddr);
        else TC_LD32(va, taddr);
        // (first tiles of a long segment, while the TMEM load is in flight) exchange the running max with the
        // other column slices.  The slices are never more than the two TMEM buffers apart, so with >= 8 tiles
        // per exchanging segment a slice can not read a value another one published for a LATER segment.
        if (exch && t < 4) {
          // float max as an integer atomic: signed max for r >= 0, unsigned min for r < 0 (correct for any mix of signs)
          const float sh = (r >= 0.f)
              ? __int_as_float(atomicMax(reinterpret_cast<int *>(&S.rmax[trow]), __float_as_int(r)))
              : __uint_as_float(atomicMin(reinterpret_cast<unsigned int *>(&S.rmax[trow]), __float_as_uint(r)));
          if (sh > r) { r = sh; thr = r - band; pack_thr(); }
        }
        TC_WAIT_LD(va);
        if constexpr (F16) {
          static_assert(SEL_SW == 64, "one packed load per slice");
          (void)vb;
          // the slice's 64 values are in registers: hand the TMEM buffer back BEFORE reducing them, so that the MMA of
          // the tile after next starts one reduction earlier (the buffer round trip, not a pipe, bounds the kernel)
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          __syncwarp();
          if (lane == 0) mbar_arrive_u32(tempty_u32 + buf * 8);
          released = true;
          if (t >= n_full) {   // last tile of the table: columns beyond its end (stale ring data) -> 0, below every live score
            const int n_valid = (int)min((int64_t)SEL_SW, j_end - (int64_t)jb0);  // may be <= 0
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              if (2 * i >= n_valid) va[i] &= 0xffff0000u;
              if (2 * i + 1 >= n_valid) va[i] &= 0x0000ffffu;
            }
          }
          process_h(va, jb0);
          process_h(va + 16, jb0 + 32);
        } else if (t < n_full) {
#pragma unroll
          for (int c = 0; c < NCH; c += 2) {
            TC_LD32(vb, taddr + (c + 1) * 32);
            process(va, jb0 + c * 32);
            TC_WAIT_LD(vb);
            if (c + 2 < NCH) {
              TC_LD32(va, taddr + (c + 2) * 32);
            } else {
              // the slice's last values are in registers: hand the TMEM buffer back before reducing them
              asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
              __syncwarp();
              if (lane == 0) mbar_arrive_u32(tempty_u32 + buf * 8);
              released = true;
            }
            process(vb, jb0 + (c + 1) * 32);
            if (c + 2 < NCH) TC_WAIT_LD(va);
          }
        } else {  // last tile of the table: mask the columns beyond its end
          const int n_valid = (int)min((int64_t)SEL_SW, j_end - (int64_t)jb0);  // may be <= 0
#pragma unroll 1
          for (int c = 0; c < NCH; ++c) {
            if (c > 0) { TC_LD32(va, taddr + c * 32); TC_WAIT_LD(va); }
            mask_tail(va, c * 32, n_valid);
            process(va, jb0 + c * 32);
          }
        }
        if (!released) {   // (tail tile of the tf32 filter)
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          __syncwarp();
          if (lane == 0) mbar_arrive_u32(tempty_u32 + buf * 8);
        }
        if (threadIdx.x == 64 && gt >= 40 && gt < 44) TC_TRACE(6 + 2 * (gt - 40));
      }
      if (live) {
        // hand the surviving chunks of this (slot, slice) stream to the refine kernel
        const int64_t stream = (int64_t)ch * slots_max * SEL_SLICES +
                               (int64_t)((int)blockIdx.x - tc_cta_of((int64_t)rt * Tch, n_units, gridDim.x)) * SEL_SLICES + slice;
        int k = 0;
        for (int e = 0; e < cnt; ++e) {
          const unsigned long long ent = list[e * TC_BM];
          if (__uint_as_float((uint32_t)(ent >> 32)) >= thr) {
            if (k < TC_OUT) out_ent[(stream * TC_OUT + k) * M + row] = ent;
            else spill(ent);
            ++k;
          }
        }
        out_r[stream * M + row] = r;
        out_cnt[stream * M + row] = (ovf || flag_all) ? -1 : min(k, TC_OUT);
      }
      if (threadIdx.x == 64) TC_TRACE(13);
    }
    }
  }

#undef TC_SEGMENT
#undef TC_CHUNK
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __threadfence_block();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem));
    if (lane == 0) TC_TRACE(14);
  }
  // Exact re-score of the chunks this CTA spilled (normally none); kept out of line so that the hot loop's
  // code layout does not depend on it
  const unsigned int n_ovf = min(S.ovf_n, ovf_cta_cap);
  if (n_ovf) tc_rescore_overflow<D>(W, n_rows, Q, ovf_ent + (size_t)blockIdx.x * ovf_cta_cap, ovf_row + (size_t)blockIdx.x * ovf_cta_cap, n_ovf, row_best);
}

#ifdef PCV_TC_TRACE
extern "C" int pcv_debug_tc_trace(long long *host16) {
  return (int)cudaMemcpyFromSymbol(host16, g_tc_trace, sizeof(long long) * 16);
}
extern "C" int pcv_debug_tc_mma(long long *host16) {
  return (int)cudaMemcpyFromSymbol(host16, g_tc_mma, sizeof(long long) * 16);
}
extern "C" int pcv_debug_tc_cta(long long *host4x256) {
  return (int)cudaMemcpyFromSymbol(host4x256, g_tc_cta, sizeof(long long) * 4 * 256);
}
#endif

// Exact refine: one warp per query row.  R = max over the row's streams of their approximate
// running maxima; every recorded chunk whose approximate maximum is >= R - band is re-scored
// item by item (lane = item) with the exact fp32 sequential-k FMA chain (SURVEY F3); winner =
// largest exact score, ties -> lowest index (SURVEY F2).  Streams flagged -1 (too many chunks
// inside the band, i.e. heavy exact ties) are scanned completely.  A row's streams are
// (column chunk, CTA slot, column slice): slot = position among the CTAs that touched the row tile in that chunk.
// (256, 5): 48 registers -> 40 resident warps per SM, so M = 10240 rows finish in two waves instead of three
template <int D>
__global__ void __launch_bounds__(256, D <= 16 ? 5 : 4)
tc_refine_kernel(const float *__restrict__ W, int64_t n_rows, int64_t row_offset, const float *__restrict__ Q,
                 int64_t M, int T, int Tc, int row_tiles, int slots_max, int G, const float *__restrict__ max_row_norm,
                 float band_const,
                 const float *__restrict__ out_r, const int32_t *__restrict__ out_cnt,
                 const unsigned long long *__restrict__ out_ent, unsigned long long *__restrict__ row_best,
                 unsigned int *__restrict__ ovf_count_reset, int64_t *__restrict__ out_idx,
                 float *__restrict__ out_val) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const int64_t rt = row / TC_BM;
  const int n_chunks = (T + Tc - 1) / Tc;
  // geometry of column chunk ch for this row tile: first CTA that touched it, number of streams, first stream id
  auto chunk_geom = [&](int ch, int &Tch, int64_t &n_units, int &cfirst, int &n_streams, int64_t &sbase) {
    Tch = min(Tc, T - ch * Tc);
    n_units = (int64_t)row_tiles * Tch;
    cfirst = tc_cta_of(rt * Tch, n_units, G);
    const int clast = tc_cta_of((rt + 1) * Tch - 1, n_units, G);
    n_streams = (clast - cfirst + 1) * SEL_SLICES;
    sbase = (int64_t)ch * slots_max * SEL_SLICES;
  };
  auto load_group = [&](int64_t sbase, int n_streams, int base, int &cnt, unsigned long long (&ents)[TC_OUT]) {
    const int s = base + lane;
    cnt = 0;
#pragma unroll
    for (int e = 0; e < TC_OUT; ++e) ents[e] = 0ull;
    if (s < n_streams) {
      cnt = out_cnt[(sbase + s) * M + row];
#pragma unroll
      for (int e = 0; e < TC_OUT; ++e) ents[e] = out_ent[((sbase + s) * TC_OUT + e) * M + row];   // e >= cnt: stale, ignored
    }
  };
  // issue every independent load before the first use: the first chunk's running maxima and lists, the query
  // row and the row's overflow winner all arrive in ONE memory round trip
  int Tch, cfirst, n_streams;
  int64_t n_units, sbase;
  chunk_geom(0, Tch, n_units, cfirst, n_streams, sbase);
  int cnt;
  unsigned long long ents[TC_OUT];
  float R = (lane < n_streams) ? out_r[(sbase + lane) * M + row] : -INFINITY;
  load_group(sbase, n_streams, 0, cnt, ents);
  const float4 q0 = __ldg(reinterpret_cast<const float4 *>(Q + row * D));
  const float4 q1 = __ldg(reinterpret_cast<const float4 *>(Q + row * D) + 1);
  const unsigned long long pb = row_best[row];   // exact winner among the overflow chunks (0 = none)
  for (int s = lane + 32; s < n_streams; s += 32) R = fmaxf(R, out_r[(sbase + s) * M + row]);
  for (int ch = 1; ch < n_chunks; ++ch) {
    int Tx, cf, ns;
    int64_t nu, sb;
    chunk_geom(ch, Tx, nu, cf, ns, sb);
    for (int s = lane; s < ns; s += 32) R = fmaxf(R, out_r[(sb + s) * M + row]);
  }
  float q[8];   // D = 8: the whole query row lives in registers; larger D re-reads it (L1 broadcast) per re-scored item
  q[0] = q0.x; q[1] = q0.y; q[2] = q0.z; q[3] = q0.w; q[4] = q1.x; q[5] = q1.y; q[6] = q1.z; q[7] = q1.w;
  float ss = 0.f;
  if constexpr (D == 8) {
#pragma unroll
    for (int k = 0; k < 8; ++k) ss = fmaf(q[k], q[k], ss);
  } else {
    ss = tc_norm2<D>(Q + row * D);
  }
  // (f16 filter: the running maxima and the recorded approximate maxima live in the scaled, shifted domain of that
  // filter, where the band is a constant)
  const float band = band_const > 0.f ? band_const : tc_band_scale(false, __ldg(max_row_norm)) * tc_norm<D>(Q + row * D, ss) * 1.0001f + 1e-37f;
  R = warp_max(R);
  const float thr = R - band;
  // R = +inf (a score overflowed) or a NaN band: the band says nothing, every stream of the row is scanned exactly
  const bool exact_row = !(thr < INFINITY);
  float best = -INFINITY;
  int32_t bidx = 0x7fffffff;
  auto score = [&](int64_t j) {
    float s = 0.f;
    if constexpr (D == 8) {
      const float4 w0 = __ldg(reinterpret_cast<const float4 *>(W + j * D));
      const float4 w1 = __ldg(reinterpret_cast<const float4 *>(W + j * D) + 1);
      s = fmaf(q[0], w0.x, s); s = fmaf(q[1], w0.y, s); s = fmaf(q[2], w0.z, s); s = fmaf(q[3], w0.w, s);
      s = fmaf(q[4], w1.x, s); s = fmaf(q[5], w1.y, s); s = fmaf(q[6], w1.z, s); s = fmaf(q[7], w1.w, s);
    } else {
      s = tc_exact_score<D>(Q + row * D, W + j * D);
    }
    if (s > best || (s == best && (int32_t)j < bidx)) { best = s; bidx = (int32_t)j; }
  };
  // lane = stream while the lists are inspected, lane = item while a chunk is re-scored
  for (int ch = 0; ch < n_chunks; ++ch) {
    if (ch > 0) chunk_geom(ch, Tch, n_units, cfirst, n_streams, sbase);
    for (int base = 0; base < n_streams; base += 32) {
      if (base > 0 || ch > 0) load_group(sbase, n_streams, base, cnt, ents);
      unsigned flagged = __ballot_sync(0xffffffffu, (cnt < 0 || exact_row) && base + lane < n_streams);
      while (flagged) {  // exact scan of a flagged stream's whole column range
        const int fs = base + __ffs(flagged) - 1;
        flagged &= flagged - 1;
        const int slot = fs / SEL_SLICES, slice = fs % SEL_SLICES;
        const int64_t c = cfirst + slot;
        const int64_t tb = max(tc_cta_begin(c, n_units, G), rt * Tch) - rt * Tch;
        const int64_t te = min(tc_cta_begin(c + 1, n_units, G), (rt + 1) * Tch) - rt * Tch;
        const int64_t j_begin = ((int64_t)ch * Tc + tb) * TC_BN;
        const int64_t j_end = min(n_rows, ((int64_t)ch * Tc + te) * TC_BN);
        for (int64_t t0 = j_begin + slice * SEL_SW; t0 < j_end; t0 += TC_BN)
          for (int i = lane; i < SEL_SW; i += 32)
            if (t0 + i < j_end) score(t0 + i);
      }
#pragma unroll
      for (int e = 0; e < TC_OUT; ++e) {
        const bool pass = (e < cnt) && __uint_as_float((uint32_t)(ents[e] >> 32)) >= thr;
        unsigned live = __ballot_sync(0xffffffffu, pass);
        while (live) {
          const int src = __ffs(live) - 1;
          live &= live - 1;
          const int64_t j = (int64_t)__shfl_sync(0xffffffffu, (uint32_t)ents[e], src) + lane;
          if (j < n_rows) score(j);
        }
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int32_t oi = __shfl_xor_sync(0xffffffffu, bidx, o);
    if (ov > best || (ov == best && oi < bidx)) { best = ov; bidx = oi; }
  }
  if (lane == 0) {
    row_best[row] = 0ull;                          // leave the workspace zeroed for the next call
    if (row == 0) *ovf_count_reset = 0u;
    if (pb) {
      float ov;
      int32_t oi;
      unpack_best(pb, &ov, &oi);
      if (ov > best || (ov == best && oi < bidx)) { best = ov; bidx = oi; }
    }
    if (bidx == 0x7fffffff) bidx = 0;   // no score above -inf (NaN never wins): the first index, value -inf
    out_idx[row] = (int64_t)bidx + row_offset;
    if (out_val) out_val[row] = best;
  }
}

// ------------------------------------------------------------------ host side
struct TcPlan {
  int row_tiles, T, grid, slots;   // T = table tiles per row tile; slots = max CTAs touching one row tile (per column chunk)
  int Tc, n_chunks;                // column chunks of Tc tiles (catalogs beyond the L2: see the kernel)
  int64_t n_units;
  unsigned int ovf_cap;
  int64_t rows_per_launch;   // rows handled per kernel triple; larger M is processed in groups
  size_t var_bytes;          // per-group part of the workspace (lists, overflow buffer)
  size_t ws_bytes;           // 256 (counter) + rows_per_launch * 8 (row_best) + max var_bytes over the groups
};

constexpr size_t TC_WS_CAP = 1536ull << 20;  // workspace budget: bigger problems are split into row groups

static void tc_plan_rows(const Table *t, int64_t M, TcPlan *p) {
  p->rows_per_launch = M;
  p->row_tiles = (int)((M + TC_BM - 1) / TC_BM);
  p->T = (int)((t->n_rows + TC_BN - 1) / TC_BN);
  p->n_units = (int64_t)p->row_tiles * p->T;
  int64_t g = p->n_units / 8;   // keep >= 8 tiles per CTA to amortise the prologue
  if (g < 1) g = 1;
  if (g > t->sm_count) g = t->sm_count;
  p->grid = (int)g;
  // column chunks: one chunk while the table (T tiles of 8 KB) fits comfortably in the 126 MB L2, else 32 MB chunks
  p->Tc = (p->T <= t->tc_chunk_tiles + t->tc_chunk_tiles / 2) ? p->T : t->tc_chunk_tiles;
  p->n_chunks = (p->T + p->Tc - 1) / p->Tc;
  int slots = 1;
  for (int ch = 0; ch < p->n_chunks; ch += (p->n_chunks > 1 ? p->n_chunks - 1 : 1)) {   // the full-size and the last chunk
    const int Tch = (p->T - ch * p->Tc < p->Tc) ? (p->T - ch * p->Tc) : p->Tc;
    const int64_t nu = (int64_t)p->row_tiles * Tch;
    for (int64_t rt = 0; rt < p->row_tiles; ++rt) {
      const int n = tc_cta_of((rt + 1) * Tch - 1, nu, p->grid) - tc_cta_of(rt * Tch, nu, p->grid) + 1;
      if (n > slots) slots = n;
    }
  }
  p->slots = slots;
  // per (stream, row): running max (4) + count (4) + TC_OUT recorded chunks (8 each);
  // per row: packed overflow winner (8); overflow list: ovf_cap x (8 + 4), split evenly over the CTAs
  const size_t n_sr = (size_t)SEL_SLICES * p->slots * p->n_chunks * (size_t)M;
  p->ovf_cap = (unsigned int)(n_sr / 16 < 65536 ? 65536 : (n_sr / 16 > (1u << 24) ? (1u << 24) : n_sr / 16));
  p->var_bytes = n_sr * (8 + 8 * TC_OUT) + (size_t)p->ovf_cap * 12;
  p->ws_bytes = 256 + (size_t)M * 8 + p->var_bytes;
}

static void tc_plan(const Table *t, int64_t M, TcPlan *p) {
  int64_t mc = M;
  tc_plan_rows(t, mc, p);
  while (p->ws_bytes > TC_WS_CAP && mc > TC_BM) {   // halve the row group until the workspace fits the budget
    mc = ((mc + 1) / 2 + TC_BM - 1) / TC_BM * TC_BM;
    tc_plan_rows(t, mc, p);
  }
  if (M % mc) {   // the shorter last group has its own partition (more slots per row tile): size for both
    TcPlan tail;
    tc_plan_rows(t, M % mc, &tail);
    if (tail.var_bytes > p->var_bytes) p->ws_bytes = 256 + (size_t)mc * 8 + tail.var_bytes;
  }
}

bool score_select_tc_supported(const Table *t) { return tc_dim_ok(t->dim) && t->tmap_valid; }

size_t score_select_tc_workspace(const Table *t, int64_t M) {
  if (!tc_dim_ok(t->dim)) return 0;
  TcPlan p;
  tc_plan(t, M, &p);
  return p.ws_bytes;
}

// Pre-swizzled image of the table (layout: sw32_chunk_index).  D = 8 (ka = 1): row j simply keeps its 32 bytes,
// chunks swapped.
__global__ void pack_sw32_kernel(const float4 *__restrict__ W, int64_t n_rows, int ka, float4 *__restrict__ out) {
  const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // 16-byte chunk index of W
  if (f >= n_rows * 2 * ka) return;
  const int64_t j = f / (2 * ka);
  const int a = (int)(f % (2 * ka)) >> 1;
  const int c = (int)(f & 1);
  out[sw32_chunk_index(j, a, c, ka)] = W[f];
}

// f16 image of a D = 8 table for the f16 filter (layout: h16_store_row)
__global__ void pack_h16_kernel(const float4 *__restrict__ W, int64_t n_rows, uint4 *__restrict__ out) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_rows) return;
  h16_store_row(out, j, W[2 * j], W[2 * j + 1]);
}

int table_init_tc(Table *t) {
  t->tmap_valid = 0;
  t->packed = nullptr;
  t->packed_h = nullptr;
  // 32 MB of the pre-swizzled table per column chunk: 4096 tiles of 8 KB at D = 8, fewer (larger) tiles beyond
  t->tc_chunk_tiles = 4096 / (t->dim >= 8 ? t->dim / 8 : 1);
  if (const char *e = getenv("PCV_TC_CHUNK_TILES")) {   // test hook: force chunking on small catalogs
    const int v = atoi(e);
    if (v >= 1) t->tc_chunk_tiles = v;
  }
  if (!tc_dim_ok(t->dim)) return PCV_OK;
  const int ka = t->dim / 8;
  // D = 8: exactly n_rows x 32 B (the last tile is copied short); D > 8: whole tiles, zero-padded
  const int64_t rows_alloc = ka == 1 ? t->n_rows : (t->n_rows + TC_BN - 1) / TC_BN * TC_BN;
  const size_t packed_bytes = (size_t)rows_alloc * t->dim * sizeof(float);
  float *p = nullptr;
  cudaError_t e = cudaMalloc(&p, packed_bytes);
  if (e != cudaSuccess) {   // no silent downgrade to the 8x slower SIMT engine: the caller sees the failure
    cudaGetLastError();
    set_error("pcv_table_create: cudaMalloc of the pre-swizzled table copy (%zu bytes) -> %s", packed_bytes,
              cudaGetErrorString(e));
    return PCV_ERR_CUDA;
  }
  if (ka > 1) cudaMemset(p, 0, packed_bytes);
  const int64_t chunks = t->n_rows * 2 * ka;
  pack_sw32_kernel<<<(unsigned)((chunks + 255) / 256), 256>>>(reinterpret_cast<const float4 *>(t->W), t->n_rows, ka,
                                                              reinterpret_cast<float4 *>(p));
  count_launch();
  e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    cudaGetLastError();
    cudaFree(p);
    set_error("pcv_table_create: packing the pre-swizzled table copy -> %s", cudaGetErrorString(e));
    return PCV_ERR_CUDA;
  }
  t->packed = p;
  t->tmap_valid = 1;
  // f16 filter image (D = 8, row norms that f16 products can carry): built eagerly, so that the first select call may
  // already be inside a CUDA graph capture
  if (t->dim == 8 && t->max_row_norm > 0.f && t->max_row_norm < 1.0e4f) {
    void *ph = nullptr;
    e = cudaMalloc(&ph, (size_t)t->n_rows * 32);
    if (e == cudaSuccess) {
      pack_h16_kernel<<<(unsigned)((t->n_rows + 255) / 256), 256>>>(reinterpret_cast<const float4 *>(t->W), t->n_rows,
                                                                    reinterpret_cast<uint4 *>(ph));
      count_launch();
      e = cudaDeviceSynchronize();
    }
    if (e != cudaSuccess) {
      cudaGetLastError();
      if (ph) cudaFree(ph);
      set_error("pcv_table_create: f16 table image -> %s", cudaGetErrorString(e));
      return PCV_ERR_CUDA;
    }
    t->packed_h = ph;
  }
  return PCV_OK;
}

void table_free_tc(Table *t) {
  if (t->packed) cudaFree(t->packed);
  t->packed = nullptr;
  if (t->packed_h) cudaFree(t->packed_h);
  t->packed_h = nullptr;
}

void launch_select_finalize(const float *pv, const int32_t *pi, int n_parts, int64_t M, int64_t row_offset,
                            int64_t *out_idx, float *out_val, cudaStream_t st);

template <int KA, bool F16 = false>
static int score_select_tc_impl(const Table *t, const float *Q, int64_t M, int64_t *out_idx, float *out_val, void *ws,
                                size_t ws_bytes, cudaStream_t st) {
  constexpr int D = 8 * KA;
  TcPlan p;
  tc_plan(t, M, &p);
  if (ws == nullptr || ws_bytes < p.ws_bytes) {
    set_error("score_select(tcgen05): workspace too small (%zu < %zu)", ws_bytes, p.ws_bytes);
    return PCV_ERR_WORKSPACE;
  }
  const int64_t Mg = p.rows_per_launch;                                // rows per group (== M when it fits)
  // fixed head (zero on entry, re-zeroed by tc_refine_kernel): a spare counter word, per-row overflow winner
  unsigned int *ovf_count = reinterpret_cast<unsigned int *>(ws);
  unsigned long long *row_best = reinterpret_cast<unsigned long long *>(static_cast<char *>(ws) + 256);   // [Mg]
  unsigned long long *var = row_best + Mg;                             // per-group layout below
  const size_t smem = sizeof(TcSmem<KA>) + 1024;
  static bool attr_set[64] = {false};
  if (!attr_set[t->device & 63]) {
    PCV_CUDA((cudaFuncSetAttribute(score_select_tc_kernel<KA, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)));
    attr_set[t->device & 63] = true;
  }
  // |tf32 chain - fp32 chain| <= 1.25 * 2^-9 * |q| * max|w|; the band is twice that.  The f16 filter gets max|w| (+0.3 %)
  // instead: it scales every query row into a fixed range, where its band is the constant TC_H_BAND.  Both kernels read
  // max|w| from the handle's device scalar (tc_band_scale), so a refresh on the stream reaches a captured graph too
  const float *wmax = t->max_row_norm_dev();
  const float *Wsw = F16 ? reinterpret_cast<const float *>(t->packed_h) : t->packed;
  for (int64_t r0 = 0; r0 < M; r0 += Mg) {   // row groups reuse the workspace back to back on the stream
    const int64_t m = (M - r0 < Mg) ? (M - r0) : Mg;
    const float *Qg = Q + r0 * D;
    // row_best / ovf_count are zero on entry: the workspace must be zero-initialised ONCE by the caller
    // (see pcv_score_select_workspace_bytes) and tc_refine_kernel re-zeroes what a call dirtied
    TcPlan g;   // the last group may be shorter: its own partition
    tc_plan_rows(t, m, &g);
    const size_t n_sr = (size_t)SEL_SLICES * g.slots * g.n_chunks * (size_t)m;   // (stream, row) pairs of this group
    unsigned long long *ent = var;                                     // [n_sr][TC_OUT]
    unsigned long long *ovf_ent = ent + n_sr * TC_OUT;                 // [ovf_cap]
    float *rr = reinterpret_cast<float *>(ovf_ent + g.ovf_cap);        // [n_sr]
    int32_t *cc = reinterpret_cast<int32_t *>(rr + n_sr);              // [n_sr]
    int32_t *ovf_row = cc + n_sr;                                      // [ovf_cap]
    score_select_tc_kernel<KA, F16><<<(unsigned)g.grid, SEL_THREADS, smem, st>>>(Wsw, t->W, t->n_rows, Qg, m, g.T, g.Tc, g.row_tiles,
                                                                       g.slots, wmax, rr, cc, ent, row_best, ovf_ent,
                                                                       ovf_row, g.ovf_cap / (unsigned)g.grid);
    PCV_LAUNCH_CHECK();
    tc_refine_kernel<D><<<(unsigned)((m + 7) / 8), 256, 0, st>>>(t->W, t->n_rows, t->row_offset, Qg, m, g.T, g.Tc, g.row_tiles,
                                                             g.slots, g.grid, wmax, F16 ? TC_H_BAND : 0.f, rr, cc, ent, row_best, ovf_count, out_idx + r0,
                                                             out_val ? out_val + r0 : nullptr);
    if (cudaPeekAtLastError() != cudaSuccess) {
      // the filter ran but the kernel that re-zeroes the head did not launch: heal the workspace here, so that a
      // failed call never poisons the next one (steady state pays nothing for this)
      cudaError_t le = cudaGetLastError();
      cudaMemsetAsync(ws, 0, 256 + (size_t)Mg * 8, st);
      set_error("score_select(tcgen05): refine kernel launch -> %s (workspace head re-zeroed)", cudaGetErrorString(le));
      return PCV_ERR_CUDA;
    }
    count_launch();
  }
  return PCV_OK;
}

bool score_select_tc_f16_supported(const Table *t) { return t->dim == 8 && t->tmap_valid && t->packed_h != nullptr; }

int score_select_tc(const Table *t, const float *Q, int64_t M, int64_t *out_idx, float *out_val, void *ws,
                    size_t ws_bytes, cudaStream_t st, int f16) {
  if (f16) {
    if (!score_select_tc_f16_supported(t)) {
      set_error("score_select(tcgen05 f16): needs dim 8 and a table whose row norms fit f16 (dim %d, max|w| %g)", t->dim, (double)t->max_row_norm);
      return PCV_ERR_UNSUPPORTED;
    }
    return score_select_tc_impl<1, true>(t, Q, M, out_idx, out_val, ws, ws_bytes, st);
  }
  switch (t->dim) {
    case 8: return score_select_tc_impl<1>(t, Q, M, out_idx, out_val, ws, ws_bytes, st);
    case 16: return score_select_tc_impl<2>(t, Q, M, out_idx, out_val, ws, ws_bytes, st);
    case 32: return score_select_tc_impl<4>(t, Q, M, out_idx, out_val, ws, ws_bytes, st);
    case 64: return score_select_tc_impl<8>(t, Q, M, out_idx, out_val, ws, ws_bytes, st);
    case 128: return score_select_tc_impl<16>(t, Q, M, out_idx, out_val, ws, ws_bytes, st);
  }
  set_error("score_select(tcgen05): dim %d unsupported (8, 16, 32, 64 or 128)", t->dim);
  return PCV_ERR_UNSUPPORTED;
}

}  // namespace pcv
