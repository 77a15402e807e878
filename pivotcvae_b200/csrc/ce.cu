// ce.cu — fused streaming masked soft-max cross-entropy over the catalog:
// loss rows, log-sum-exp AND d(loss_row)/dq in one pass; the (M x N) logits,
// the Bernoulli mask and the soft-max never reach HBM.
//
// Replaces (reference file:line)
//   pivotcvae.py:274 / listcvae.py:166   p = mm(prox_emb, table.t())        (M x N, materialised)
//   train_generative.py:36-42            downsample: mask = onehot(target) U Bernoulli(n_neg/N); pred*mask
//   train_generative.py:59               CrossEntropyLoss (log-softmax + nll), and their backward
//
// Semantics kept (SURVEY F7): masked-OUT logits become 0 (not -inf):
//   lse_i  = log( sum_{j in mask_i} e^{x_ij} + (N - |mask_i|) )
//   loss_i = lse_i - x_{i,t_i}
//   dq_i   = sum_{j in mask_i} softmax_ij * w_j - w_{t_i}          (table frozen: no dW)
//
// Layout mirrors score_select.cu: CTA = 8 warps x R rows, catalog split over
// blockIdx.y, cp.async double-buffered float4-SoA tiles.  Each lane keeps an
// online-softmax state (running max m, sum l, dq accumulator) for its rows;
// lanes, then splits, are merged with the usual rescale.
#include "pcv_common.cuh"

namespace pcv {

constexpr int CE_WARPS = 8;
constexpr int CE_THREADS = CE_WARPS * 32;
constexpr int CE_TILE_FLOATS = 8192;

enum { CE_DENSE = 0, CE_BITMASK = 1 };
constexpr size_t CE_GB_HOST = 1024;  // == CE_GB (gap-process block, see ce_sparse_kernel)

template <int D>
struct CECfg {
  static constexpr int R = (D <= 8) ? 4 : (D <= 16 ? 2 : 1);
  static constexpr int ROWS = CE_WARPS * R;
  static constexpr int TILE = (CE_TILE_FLOATS / D) < 128 ? 128 : (CE_TILE_FLOATS / D);
  static constexpr int C4 = D / 4;
  static constexpr size_t SMEM = 2ull * TILE * D * sizeof(float);
};

struct CEPlan {
  int rows_per_cta, tile, row_tiles, n_split;
  int64_t items_per_split;
  int rec;  // floats per (split,row) partial record: m, l, cnt, dq[D]
  size_t ws_bytes;
};

static int ce_rows_for(int D) {
  switch (D) {
    case 4: return CECfg<4>::ROWS;
    case 8: return CECfg<8>::ROWS;
    case 16: return CECfg<16>::ROWS;
    case 32: return CECfg<32>::ROWS;
    case 64: return CECfg<64>::ROWS;
    case 128: return CECfg<128>::ROWS;
  }
  return 0;
}

static int ce_plan(const Table *t, int64_t M, CEPlan *p) {
  p->rows_per_cta = ce_rows_for(t->dim);
  if (!p->rows_per_cta) return PCV_ERR_UNSUPPORTED;
  p->tile = CE_TILE_FLOATS / t->dim < 128 ? 128 : CE_TILE_FLOATS / t->dim;
  p->row_tiles = (int)((M + p->rows_per_cta - 1) / p->rows_per_cta);
  int64_t n_tiles = (t->n_rows + p->tile - 1) / p->tile;
  int64_t want = (4LL * t->sm_count + p->row_tiles - 1) / p->row_tiles;
  int64_t max_split = (n_tiles + 3) / 4;
  if (max_split < 1) max_split = 1;
  int64_t ns = want < 1 ? 1 : (want > max_split ? max_split : want);
  int64_t tps = (n_tiles + ns - 1) / ns;
  ns = (n_tiles + tps - 1) / tps;
  p->n_split = (int)ns;
  p->items_per_split = tps * p->tile;
  p->rec = 3 + t->dim;
  p->ws_bytes = (size_t)ns * (size_t)M * p->rec * sizeof(float);
  if (p->ws_bytes < (CE_GB_HOST + 1) * sizeof(uint32_t)) p->ws_bytes = (CE_GB_HOST + 1) * sizeof(uint32_t);
  return PCV_OK;
}

__device__ __forceinline__ void ce_cp_async16(void *smem, const void *gmem, bool valid) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(sz));
}

template <int D, int MODE>
__global__ void __launch_bounds__(CE_THREADS, (D <= 64 ? 2 : 1))
ce_kernel(const float *__restrict__ W, int64_t n_rows, int64_t row_offset,
          const float *__restrict__ Q, const int64_t *__restrict__ targets, int64_t M,
          int64_t items_per_split, const uint32_t *__restrict__ bitmask, int64_t mask_words,
          uint64_t seed, uint64_t offset, const uint64_t *__restrict__ offset_dev, uint32_t thresh,
          float *__restrict__ part) {
  using Cfg = CECfg<D>;
  constexpr int R = Cfg::R, TILE = Cfg::TILE, C4 = Cfg::C4, REC = 3 + D;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float4 *tile4 = reinterpret_cast<float4 *>(smem_raw);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row0 = (int64_t)blockIdx.x * Cfg::ROWS + (int64_t)warp * R;
  const int64_t j_begin = (int64_t)blockIdx.y * items_per_split;
  const int64_t j_end = min(n_rows, j_begin + items_per_split);
  const int n_tiles = (int)((j_end - j_begin + TILE - 1) / TILE);

  float q[R][D];
  int64_t tgt[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const bool ok = (row0 + r) < M;
    tgt[r] = ok ? targets[row0 + r] - row_offset : -1;
#pragma unroll
    for (int c = 0; c < C4; ++c) {
      float4 v = ok ? __ldg(reinterpret_cast<const float4 *>(Q + (row0 + r) * D) + c)
                    : make_float4(0.f, 0.f, 0.f, 0.f);
      q[r][4 * c + 0] = v.x; q[r][4 * c + 1] = v.y; q[r][4 * c + 2] = v.z; q[r][4 * c + 3] = v.w;
    }
  }
  float m[R], l[R], acc[R][D];
  int cnt[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    m[r] = -INFINITY; l[r] = 0.f; cnt[r] = 0;
#pragma unroll
    for (int k = 0; k < D; ++k) acc[r][k] = 0.f;
  }

  auto load_tile = [&](int t, int buf) {
    const int64_t base = j_begin + (int64_t)t * TILE;
    float4 *dst = tile4 + (size_t)buf * C4 * TILE;
    const float4 *src = reinterpret_cast<const float4 *>(W + base * D);
#pragma unroll 4
    for (int f = threadIdx.x; f < TILE * C4; f += CE_THREADS) {
      int item = f / C4, c = f % C4;
      bool valid = (base + item) < j_end;
      ce_cp_async16(dst + c * TILE + item, valid ? (const void *)(src + f) : (const void *)W, valid);
    }
    asm volatile("cp.async.commit_group;\n" ::);
  };

  if (n_tiles > 0) load_tile(0, 0);
  for (int t = 0; t < n_tiles; ++t) {
    if (t + 1 < n_tiles) {
      load_tile(t + 1, (t + 1) & 1);
      asm volatile("cp.async.wait_group 1;\n" ::);
    } else {
      asm volatile("cp.async.wait_group 0;\n" ::);
    }
    __syncthreads();
    const float4 *cur = tile4 + (size_t)(t & 1) * C4 * TILE;
    const int64_t base = j_begin + (int64_t)t * TILE;
    const int n_valid = (int)min((int64_t)TILE, j_end - base);
    for (int i = lane; i < n_valid; i += 32) {
      const int64_t j = base + i;
      bool in[R];
      bool any = false;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        bool b;
        if (MODE == CE_DENSE) {
          b = true;
        } else {
          // base and i-lane are multiples of 32: the warp shares one word per row
          uint32_t word = (row0 + r < M) ? __ldg(bitmask + (row0 + r) * mask_words + (j >> 5)) : 0u;
          b = (word >> (j & 31)) & 1u;
        }
        b = b || (j == tgt[r]);
        in[r] = b;
        any = any || b;
      }
      if (!any) continue;
      float w[D];
#pragma unroll
      for (int c = 0; c < C4; ++c) {
        const float4 v = cur[c * TILE + i];
        w[4 * c + 0] = v.x; w[4 * c + 1] = v.y; w[4 * c + 2] = v.z; w[4 * c + 3] = v.w;
      }
#pragma unroll
      for (int r = 0; r < R; ++r) {
        if (!in[r]) continue;
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < D; ++k) s = fmaf(q[r][k], w[k], s);
        cnt[r] += 1;
        if (s > m[r]) {
          const float sc = __expf(m[r] - s);  // m=-inf -> 0
          l[r] *= sc;
#pragma unroll
          for (int k = 0; k < D; ++k) acc[r][k] *= sc;
          m[r] = s;
        }
        const float p = __expf(s - m[r]);
        l[r] += p;
#pragma unroll
        for (int k = 0; k < D; ++k) acc[r][k] = fmaf(p, w[k], acc[r][k]);
      }
    }
    __syncthreads();
  }

  // merge lanes (rescale to the common max)
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const float mw = warp_max(m[r]);
    const float sc = (m[r] == -INFINITY) ? 0.f : __expf(m[r] - mw);
    float lw = warp_sum(l[r] * sc);
    int cw = cnt[r];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cw += __shfl_xor_sync(0xffffffffu, cw, o);
    float a[D];
#pragma unroll
    for (int k = 0; k < D; ++k) a[k] = warp_sum(acc[r][k] * sc);
    if (lane == 0 && row0 + r < M) {
      float *rec = part + ((int64_t)blockIdx.y * M + row0 + r) * REC;
      rec[0] = mw; rec[1] = lw; rec[2] = __int_as_float(cw);
#pragma unroll
      for (int k = 0; k < D; ++k) rec[3 + k] = a[k];
    }
  }
}

// One WARP per row: lanes walk the row's partial records (lane = record, 32 at a time), each record's weight
// e^{m - M} is computed once, and the max / sums are warp reductions in a fixed order (deterministic).  Adds the
// masked-out mass, emits loss / lse / dq; the target logit is re-derived with the exact FMA chain.
// rec_out != NULL (vocab-parallel shard): hand out the merged partial {m, l, acc[D]} of this shard's columns
// instead (no target terms); pcv_ce_vp_merge combines the shards' records after the all-gather.
__global__ void __launch_bounds__(256)
ce_finalize_kernel(const float *__restrict__ part, int n_split, int64_t M, int D,
                   const float *__restrict__ W, int64_t n_rows, int64_t row_offset,
                   const float *__restrict__ Q, const int64_t *__restrict__ targets,
                   float *__restrict__ loss_rows, float *__restrict__ lse_out,
                   float *__restrict__ dq, float *__restrict__ rec_out) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (i >= M) return;
  const int REC = 3 + D;
  float mx = -INFINITY;
  int cnt_l = 0;
  for (int s = lane; s < n_split; s += 32) {
    const float *rec = part + ((int64_t)s * M + i) * REC;
    mx = fmaxf(mx, rec[0]);
    cnt_l += __float_as_int(rec[2]);
  }
  mx = warp_max(mx);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt_l += __shfl_xor_sync(0xffffffffu, cnt_l, o);
  const int64_t n_out = n_rows - cnt_l;  // masked-out logits are exactly 0
  if (n_out > 0) mx = fmaxf(mx, 0.f);
  // lane accumulates the dq components k = lane, lane + 32, lane + 64, lane + 96 (D <= 128); every lane needs every record's weight:
  // records are processed in groups of 32 (lane = record), the group's weights are broadcast with shuffles
  float L = 0.f, acc = 0.f, acc2 = 0.f, acc3 = 0.f, acc4 = 0.f;
  if (D <= 16) {
    // small D (every BASELINE config: D = 8): lane = record keeps its own D scaled components (all loads independent,
    // one round trip), then D warp sums; lane k ends up holding component k
    float a[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) a[k] = 0.f;
    for (int s = lane; s < n_split; s += 32) {
      const float *rec = part + ((int64_t)s * M + i) * REC;
      if (rec[0] != -INFINITY) {
        const float wgt = __expf(rec[0] - mx);
        L += rec[1] * wgt;
#pragma unroll
        for (int k = 0; k < 16; ++k)
          if (k < D) a[k] = fmaf(rec[3 + k], wgt, a[k]);
      }
    }
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float t = warp_sum(a[k]);
      if (lane == k) acc = t;
    }
  } else
  for (int base = 0; base < n_split; base += 32) {
    const int s = base + lane;
    float wgt = 0.f, l_s = 0.f;
    const float *rec = part + ((int64_t)min(s, n_split - 1) * M + i) * REC;
    if (s < n_split && rec[0] != -INFINITY) {
      wgt = __expf(rec[0] - mx);
      l_s = rec[1];
    }
    L += l_s * wgt;
    const int n_here = min(32, n_split - base);
    for (int j = 0; j < n_here; ++j) {
      const float wj = __shfl_sync(0xffffffffu, wgt, j);
      if (wj != 0.f) {
        const float *rj = part + ((int64_t)(base + j) * M + i) * REC + 3;
        if (lane < D) acc = fmaf(rj[lane], wj, acc);
        if (lane + 32 < D) acc2 = fmaf(rj[lane + 32], wj, acc2);
        if (lane + 64 < D) acc3 = fmaf(rj[lane + 64], wj, acc3);
        if (lane + 96 < D) acc4 = fmaf(rj[lane + 96], wj, acc4);
      }
    }
  }
  L = warp_sum(L);
  L += (float)n_out * __expf(-mx);
  if (rec_out) {
    float *o = rec_out + i * (2 + D);
    if (lane == 0) { o[0] = mx; o[1] = L; }
    if (lane < D) o[2 + lane] = acc;
    if (lane + 32 < D) o[2 + lane + 32] = acc2;
    if (lane + 64 < D) o[2 + lane + 64] = acc3;
    if (lane + 96 < D) o[2 + lane + 96] = acc4;
    return;
  }
  const float lse = mx + logf(L);
  const int64_t t = targets[i] - row_offset;
  const float *wt = W + t * D;
  const float *qi = Q + i * D;
  if (lane == 0) {
    float xt = 0.f;
    for (int k = 0; k < D; ++k) xt = fmaf(qi[k], wt[k], xt);
    if (loss_rows) loss_rows[i] = lse - xt;
    if (lse_out) lse_out[i] = lse;
  }
  if (dq && lane < D) dq[i * D + lane] = acc * (1.f / L) - wt[lane];
  if (dq && lane + 32 < D) dq[i * D + lane + 32] = acc2 * (1.f / L) - wt[lane + 32];
  if (dq && lane + 64 < D) dq[i * D + lane + 64] = acc3 * (1.f / L) - wt[lane + 64];
  if (dq && lane + 96 < D) dq[i * D + lane + 96] = acc4 * (1.f / L) - wt[lane + 96];
}

// Vocab-parallel merge (SURVEY §8e): recs = [G][M][2 + D] shard records {m, l, acc[D]} in any shard order
// (the combination is symmetric); W is the WHOLE fp32 table (every rank keeps it: <= 320 MB), so the target logit
// and the target row come from the exact chain as in the single-GPU finalize.
__global__ void ce_vp_merge_kernel(const float *__restrict__ recs, int G, int64_t M, int D, const float *__restrict__ W,
                                   const float *__restrict__ Q, const int64_t *__restrict__ targets,
                                   float *__restrict__ loss_rows, float *__restrict__ lse_out, float *__restrict__ dq) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  const int REC = 2 + D;
  float mx = -INFINITY;
  for (int g = 0; g < G; ++g) mx = fmaxf(mx, recs[((int64_t)g * M + i) * REC]);
  float L = 0.f;
  for (int g = 0; g < G; ++g) {
    const float *rec = recs + ((int64_t)g * M + i) * REC;
    if (rec[0] != -INFINITY) L += rec[1] * __expf(rec[0] - mx);
  }
  const float lse = mx + logf(L);
  const float *wt = W + targets[i] * D;
  const float *qi = Q + i * D;
  float xt = 0.f;
  for (int k = 0; k < D; ++k) xt = fmaf(qi[k], wt[k], xt);
  if (loss_rows) loss_rows[i] = lse - xt;
  if (lse_out) lse_out[i] = lse;
  if (dq) {
    const float inv = 1.f / L;
    for (int k = 0; k < D; ++k) {
      float a = 0.f;
      for (int g = 0; g < G; ++g) {
        const float *rec = recs + ((int64_t)g * M + i) * REC;
        if (rec[0] != -INFINITY) a += rec[2 + k] * __expf(rec[0] - mx);
      }
      dq[i * D + k] = a * inv - wt[k];
    }
  }
}

// ---------------------------------------------------------------------------
// Sparse masked CE (keep_prob < 1, Philox mode): the Bernoulli(keep) mask of
// train_generative.py:39 is generated as a GAP PROCESS — inside every block of
// CE_GB consecutive columns the distance to the next kept column is Geometric(keep)
// (memoryless, so the columns are exactly i.i.d. Bernoulli(keep)) — and only the
// kept columns (~keep*N per row, 1000 of 100k by default) are ever touched:
// gather the 32-byte row, exact FMA-chain logit, online soft-max, dq accumulate.
// Work per row is O(n_neg) instead of O(N).  Gaps come from an integer inverse-CDF
// table T[g] = floor((1-keep)^g * 2^32) built by an exact 64-bit recurrence, so the
// mask is reproduced bit for bit by the CPU oracle (no transcendental involved).
// One warp per row; lane = gap-process block (round-robin).
// ---------------------------------------------------------------------------
constexpr int CE_GB = 1024;   // columns per gap-process block

__global__ void ce_gap_table_kernel(uint32_t q32, uint32_t *__restrict__ T) {
  // T[g] = P(gap >= g) * 2^32 for g = 1..CE_GB; q32 = round((1 - keep) * 2^32); T[0] unused (= 2^32)
  unsigned long long t = 0x100000000ull;
  T[0] = 0xffffffffu;
  for (int g = 1; g <= CE_GB; ++g) {
    t = (t * (unsigned long long)q32) >> 32;
    T[g] = (uint32_t)t;
  }
}

// number of g in [1, CE_GB] with u < T[g]  (T is non-increasing) == the gap length, CE_GB = "past the block"
__device__ __forceinline__ int gap_from_u(const uint32_t *__restrict__ T, uint32_t u) {
  int lo = 0, hi = CE_GB;       // invariant: u < T[g] for all 1 <= g <= lo ; u >= T[g] for g > hi
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (u < __ldg(T + mid)) lo = mid; else hi = mid - 1;
  }
  return lo;
}

template <int D>
__global__ void __launch_bounds__(256)
ce_sparse_kernel(const float *__restrict__ W, int64_t n_rows, const float *__restrict__ Q,
                 const int64_t *__restrict__ targets, int64_t M, const uint32_t *__restrict__ T, uint64_t seed,
                 uint64_t offset, const uint64_t *__restrict__ offset_dev, float *__restrict__ loss_rows,
                 float *__restrict__ lse_out, float *__restrict__ dq) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  if (offset_dev) offset += *offset_dev;
  const uint64_t rr = (uint64_t)row + offset;
  float q[D];
#pragma unroll
  for (int c = 0; c < D / 4; ++c) {
    const float4 v = __ldg(reinterpret_cast<const float4 *>(Q + row * D) + c);
    q[4 * c] = v.x; q[4 * c + 1] = v.y; q[4 * c + 2] = v.z; q[4 * c + 3] = v.w;
  }
  const int64_t tgt = targets[row];
  float m = -INFINITY, l = 0.f, acc[D];
#pragma unroll
  for (int k = 0; k < D; ++k) acc[k] = 0.f;
  int cnt = 0;
  bool seen_tgt = false;
  auto visit = [&](int64_t j) {
    float w[D];
#pragma unroll
    for (int c = 0; c < D / 4; ++c) {
      const float4 v = __ldg(reinterpret_cast<const float4 *>(W + j * D) + c);
      w[4 * c] = v.x; w[4 * c + 1] = v.y; w[4 * c + 2] = v.z; w[4 * c + 3] = v.w;
    }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < D; ++k) s = fmaf(q[k], w[k], s);
    ++cnt;
    if (s > m) {
      const float sc = __expf(m - s);
      l *= sc;
#pragma unroll
      for (int k = 0; k < D; ++k) acc[k] *= sc;
      m = s;
    }
    const float p = __expf(s - m);
    l += p;
#pragma unroll
    for (int k = 0; k < D; ++k) acc[k] = fmaf(p, w[k], acc[k]);
  };
  const int64_t n_blocks = (n_rows + CE_GB - 1) / CE_GB;
  for (int64_t b = lane; b < n_blocks; b += 32) {
    int c = -1;
    Philox4 ph = {0, 0, 0, 0};
    for (int k = 0;; ++k) {
      if ((k & 3) == 0)
        ph = philox4x32_10((uint32_t)b, (uint32_t)rr, (uint32_t)(rr >> 32),
                           PCV_STREAM_BERNOULLI + ((uint32_t)(k >> 2) << 4), (uint32_t)seed, (uint32_t)(seed >> 32));
      const uint32_t u = (k & 3) == 0 ? ph.x : ((k & 3) == 1 ? ph.y : ((k & 3) == 2 ? ph.z : ph.w));
      c += 1 + gap_from_u(T, u);
      if (c >= CE_GB) break;
      const int64_t j = b * CE_GB + c;
      if (j >= n_rows) break;
      if (j == tgt) seen_tgt = true;
      visit(j);
    }
  }
  // the target column is always part of the mask (train_generative.py:38)
  const bool any_seen = __any_sync(0xffffffffu, seen_tgt);
  if (lane == 0 && !any_seen) visit(tgt);
  // merge the 32 lane states
  const float mw = warp_max(m);
  const float sc = (m == -INFINITY) ? 0.f : __expf(m - mw);
  float lw = warp_sum(l * sc);
  int cw = cnt;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cw += __shfl_xor_sync(0xffffffffu, cw, o);
  float a[D];
#pragma unroll
  for (int k = 0; k < D; ++k) a[k] = warp_sum(acc[k] * sc);
  if (lane == 0) {
    const int64_t n_out = n_rows - cw;          // masked-out logits are exactly 0 (SURVEY F7)
    const float mx = n_out > 0 ? fmaxf(mw, 0.f) : mw;
    const float resc = __expf(mw - mx);
    const float L = lw * resc + (float)n_out * __expf(-mx);
    const float lse = mx + logf(L);
    const float *wt = W + tgt * D;
    float xt = 0.f;
#pragma unroll
    for (int k = 0; k < D; ++k) xt = fmaf(q[k], wt[k], xt);
    if (loss_rows) loss_rows[row] = lse - xt;
    if (lse_out) lse_out[row] = lse;
    if (dq) {
      const float inv = resc / L;
#pragma unroll
      for (int k = 0; k < D; ++k) dq[row * D + k] = a[k] * inv - wt[k];
    }
  }
}

template <int D>
static int launch_ce_sparse(const Table *t, const float *Q, const int64_t *targets, int64_t M, const pcv_ce_mask *mask,
                            uint32_t *T, float *loss_rows, float *lse, float *dq, cudaStream_t st) {
  double qd = (1.0 - mask->keep_prob) * 4294967296.0;
  const uint32_t q32 = qd <= 0.0 ? 0u : (qd >= 4294967295.0 ? 0xffffffffu : (uint32_t)(qd + 0.5));
  ce_gap_table_kernel<<<1, 1, 0, st>>>(q32, T);
  PCV_LAUNCH_CHECK();
  ce_sparse_kernel<D><<<(unsigned)((M + 7) / 8), 256, 0, st>>>(t->W, t->n_rows, Q, targets, M, T, mask->seed,
                                                            mask->offset, mask->offset_dev, loss_rows, lse, dq);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

// ---------------------------------------------------------------------------
// Candidate-mode (sampled soft-max) cross-entropy — the reference's default training
// mode (train_generative.py:52-56; pivotcvae.py:265-271 / listcvae.py:157-163):
//   p[i, c] = <docEmbed[cand[i, c]], q_i>   (gather + bmm),   loss_i = CE(p[i, :], tgt_pos[i])
// One warp per row: lanes stride over the nC candidates, gather the 32-byte rows,
// exact FMA-chain logit, online soft-max, dq accumulate; duplicates in the candidate
// list count once per occurrence, exactly like the reference's bmm + CrossEntropyLoss.
// Optionally materialises p (forward()'s first return value).
// ---------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(256)
cand_ce_kernel(const float *__restrict__ W, const float *__restrict__ Q, const int64_t *__restrict__ cand,
               const int64_t *__restrict__ tgt_pos, int64_t M, int nC, float *__restrict__ loss_rows,
               float *__restrict__ lse_out, float *__restrict__ dq, float *__restrict__ logits_out) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  float q[D];
#pragma unroll
  for (int c = 0; c < D / 4; ++c) {
    const float4 v = __ldg(reinterpret_cast<const float4 *>(Q + row * D) + c);
    q[4 * c] = v.x; q[4 * c + 1] = v.y; q[4 * c + 2] = v.z; q[4 * c + 3] = v.w;
  }
  float m = -INFINITY, l = 0.f, acc[D];
#pragma unroll
  for (int k = 0; k < D; ++k) acc[k] = 0.f;
  const int64_t *cr = cand + row * nC;
  for (int c = lane; c < nC; c += 32) {
    const int64_t j = __ldg(cr + c);
    float w[D];
#pragma unroll
    for (int v4 = 0; v4 < D / 4; ++v4) {
      const float4 v = __ldg(reinterpret_cast<const float4 *>(W + j * D) + v4);
      w[4 * v4] = v.x; w[4 * v4 + 1] = v.y; w[4 * v4 + 2] = v.z; w[4 * v4 + 3] = v.w;
    }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < D; ++k) s = fmaf(w[k], q[k], s);   // bmm(candidateEmb, prox): row of W first
    if (logits_out) logits_out[row * nC + c] = s;
    if (s > m) {
      const float sc = __expf(m - s);
      l *= sc;
#pragma unroll
      for (int k = 0; k < D; ++k) acc[k] *= sc;
      m = s;
    }
    const float p = __expf(s - m);
    l += p;
#pragma unroll
    for (int k = 0; k < D; ++k) acc[k] = fmaf(p, w[k], acc[k]);
  }
  const float mw = warp_max(m);
  const float sc = (m == -INFINITY) ? 0.f : __expf(m - mw);
  const float L = warp_sum(l * sc);
  float a[D];
#pragma unroll
  for (int k = 0; k < D; ++k) a[k] = warp_sum(acc[k] * sc);
  if (lane == 0) {
    const float lse = mw + logf(L);
    const int64_t jt = cr[tgt_pos[row]];
    const float *wt = W + jt * D;
    float xt = 0.f;
#pragma unroll
    for (int k = 0; k < D; ++k) xt = fmaf(wt[k], q[k], xt);
    if (loss_rows) loss_rows[row] = lse - xt;
    if (lse_out) lse_out[row] = lse;
    if (dq) {
      const float inv = 1.f / L;
#pragma unroll
      for (int k = 0; k < D; ++k) dq[row * D + k] = a[k] * inv - wt[k];
    }
  }
}

template <int D, int MODE>
static int launch_ce(const Table *t, const CEPlan &p, const float *Q, const int64_t *targets,
                     int64_t M, const uint32_t *bitmask, int64_t mask_words, uint64_t seed,
                     uint64_t offset, const uint64_t *offset_dev, uint32_t thresh, float *part, cudaStream_t st) {
  using Cfg = CECfg<D>;
  auto kern = ce_kernel<D, MODE>;
  static bool attr_set[64] = {false};
  if (!attr_set[t->device & 63]) {
    PCV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM));
    attr_set[t->device & 63] = true;
  }
  dim3 grid((unsigned)p.row_tiles, (unsigned)p.n_split);
  kern<<<grid, CE_THREADS, Cfg::SMEM, st>>>(t->W, t->n_rows, t->row_offset, Q, targets, M,
                                            p.items_per_split, bitmask, mask_words, seed, offset,
                                            offset_dev, thresh, part);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

template <int MODE>
static int ce_dispatch(const Table *t, const CEPlan &p, const float *Q, const int64_t *targets,
                       int64_t M, const uint32_t *bitmask, int64_t mask_words, uint64_t seed,
                       uint64_t offset, const uint64_t *offset_dev, uint32_t thresh, float *part,
                       cudaStream_t st) {
  switch (t->dim) {
    case 4: return launch_ce<4, MODE>(t, p, Q, targets, M, bitmask, mask_words, seed, offset, offset_dev, thresh, part, st);
    case 8: return launch_ce<8, MODE>(t, p, Q, targets, M, bitmask, mask_words, seed, offset, offset_dev, thresh, part, st);
    case 16: return launch_ce<16, MODE>(t, p, Q, targets, M, bitmask, mask_words, seed, offset, offset_dev, thresh, part, st);
    case 32: return launch_ce<32, MODE>(t, p, Q, targets, M, bitmask, mask_words, seed, offset, offset_dev, thresh, part, st);
    case 64: return launch_ce<64, MODE>(t, p, Q, targets, M, bitmask, mask_words, seed, offset, offset_dev, thresh, part, st);
    case 128: return launch_ce<128, MODE>(t, p, Q, targets, M, bitmask, mask_words, seed, offset, offset_dev, thresh, part, st);
  }
  set_error("ce: dim %d unsupported (use 4, 8, 16, 32, 64 or 128)", t->dim);
  return PCV_ERR_UNSUPPORTED;
}

// tensor-core engine (ce_tc2.cu)
bool ce_tc_supported(const Table *t);
size_t ce_tc_workspace(const Table *t, int64_t M);
int ce_tc_launch(const Table *t, const float *Q, const int64_t *targets, int64_t M, float *part, size_t ws_bytes, cudaStream_t st);

}  // namespace pcv

using namespace pcv;

extern "C" {

int pcv_cand_ce_fwd_bwd(const pcv_table *th, const float *Q, const int64_t *candidates, const int64_t *target_pos,
                        int64_t M, int n_cand, float *loss_rows, float *lse, float *dq, float *logits_out,
                        pcv_stream_t stream) {
  PCV_CHECK_ARG(th && Q && candidates && target_pos, "NULL pointer");
  PCV_CHECK_ARG(M > 0 && n_cand > 0, "bad shape");
  const Table *t = reinterpret_cast<const Table *>(th);
  PCV_CHECK_ARG(t->row_offset == 0, "candidate CE needs the whole table (row_offset 0)");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned blocks = (unsigned)((M + 7) / 8);
  switch (t->dim) {
    case 4: cand_ce_kernel<4><<<blocks, 256, 0, st>>>(t->W, Q, candidates, target_pos, M, n_cand, loss_rows, lse, dq, logits_out); break;
    case 8: cand_ce_kernel<8><<<blocks, 256, 0, st>>>(t->W, Q, candidates, target_pos, M, n_cand, loss_rows, lse, dq, logits_out); break;
    case 16: cand_ce_kernel<16><<<blocks, 256, 0, st>>>(t->W, Q, candidates, target_pos, M, n_cand, loss_rows, lse, dq, logits_out); break;
    case 32: cand_ce_kernel<32><<<blocks, 256, 0, st>>>(t->W, Q, candidates, target_pos, M, n_cand, loss_rows, lse, dq, logits_out); break;
    case 64: cand_ce_kernel<64><<<blocks, 256, 0, st>>>(t->W, Q, candidates, target_pos, M, n_cand, loss_rows, lse, dq, logits_out); break;
    case 128: cand_ce_kernel<128><<<blocks, 256, 0, st>>>(t->W, Q, candidates, target_pos, M, n_cand, loss_rows, lse, dq, logits_out); break;
    default:
      set_error("cand_ce: dim %d unsupported", t->dim);
      return PCV_ERR_UNSUPPORTED;
  }
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

int pcv_ce_workspace_bytes(const pcv_table *th, int64_t M, size_t *bytes_host) {
  PCV_CHECK_ARG(th && bytes_host, "NULL pointer");
  PCV_CHECK_ARG(M > 0, "M must be > 0");
  const Table *t = reinterpret_cast<const Table *>(th);
  CEPlan p;
  if (ce_plan(t, M, &p) != PCV_OK) {
    set_error("ce: dim %d unsupported", t->dim);
    return PCV_ERR_UNSUPPORTED;
  }
  size_t b = p.ws_bytes;
  const size_t tc = ce_tc_workspace(t, M);
  if (tc > b) b = tc;
  *bytes_host = (b + 255) & ~(size_t)255;
  return PCV_OK;
}

static int ce_run(const pcv_table *th, const float *Q, const int64_t *targets, int64_t M,
                  const pcv_ce_mask *mask, float *loss_rows, float *lse, float *dq, float *rec_out,
                  void *workspace, size_t workspace_bytes, pcv_stream_t stream) {
  PCV_CHECK_ARG(th && Q && targets && mask, "NULL pointer");
  PCV_CHECK_ARG(M > 0, "M must be > 0");
  const Table *t = reinterpret_cast<const Table *>(th);
  PCV_CHECK_ARG(t->n_rows < 0x7fffffffLL, "shard larger than 2^31-1 rows");
  PCV_CHECK_ARG(rec_out != nullptr || t->row_offset == 0,
                "a table shard (row_offset > 0) yields partial records: call pcv_ce_partials + pcv_ce_vp_merge");
  PCV_CHECK_ARG(rec_out == nullptr || (mask->bitmask == nullptr && mask->keep_prob >= 1.0),
                "pcv_ce_partials serves the full-catalog soft-max (keep_prob >= 1, no bitmask); the sparse mask "
                "visits O(n_neg) columns per row and needs no sharding");
  PCV_CHECK_ARG(mask->keep_prob > 0.0, "keep_prob must be > 0");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  CEPlan p;
  if (ce_plan(t, M, &p) != PCV_OK) {
    set_error("ce: dim %d unsupported", t->dim);
    return PCV_ERR_UNSUPPORTED;
  }
  if (!workspace || (workspace_bytes < p.ws_bytes && mask->engine != PCV_CE_ENGINE_TF32)) {
    set_error("ce: workspace too small (%zu < %zu)", workspace_bytes, p.ws_bytes);
    return PCV_ERR_WORKSPACE;
  }
  float *part = reinterpret_cast<float *>(workspace);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t mask_words = (t->n_rows + 31) / 32;
  if (mask->bitmask) {
    rc = ce_dispatch<CE_BITMASK>(t, p, Q, targets, M, mask->bitmask, mask_words, 0, 0, nullptr, 0, part, st);
  } else if (mask->keep_prob >= 1.0 && mask->engine == PCV_CE_ENGINE_TF32) {
    if (!ce_tc_supported(t)) {
      set_error("ce: the tf32 engine serves dims 8, 16, 32, 64 and 128 (this table has dim %d)", t->dim);
      return PCV_ERR_UNSUPPORTED;
    }
    const int n_parts = ce_tc_launch(t, Q, targets, M, part, workspace_bytes, st);
    if (n_parts < 0) return n_parts;
    ce_finalize_kernel<<<(unsigned)((M + 7) / 8), 256, 0, st>>>(part, n_parts, M, t->dim, t->W, t->n_rows,
                                                                    t->row_offset, Q, targets, loss_rows, lse, dq, rec_out);
    PCV_LAUNCH_CHECK();
    return PCV_OK;
  } else if (mask->keep_prob >= 1.0) {
    rc = ce_dispatch<CE_DENSE>(t, p, Q, targets, M, nullptr, 0, 0, 0, nullptr, 0, part, st);
  } else {
    // sparse path: only the kept columns are visited; the workspace holds the gap table
    uint32_t *T = reinterpret_cast<uint32_t *>(workspace);
    switch (t->dim) {
      case 4: return launch_ce_sparse<4>(t, Q, targets, M, mask, T, loss_rows, lse, dq, st);
      case 8: return launch_ce_sparse<8>(t, Q, targets, M, mask, T, loss_rows, lse, dq, st);
      case 16: return launch_ce_sparse<16>(t, Q, targets, M, mask, T, loss_rows, lse, dq, st);
      case 32: return launch_ce_sparse<32>(t, Q, targets, M, mask, T, loss_rows, lse, dq, st);
      case 64: return launch_ce_sparse<64>(t, Q, targets, M, mask, T, loss_rows, lse, dq, st);
      case 128: return launch_ce_sparse<128>(t, Q, targets, M, mask, T, loss_rows, lse, dq, st);
    }
    set_error("ce: dim %d unsupported", t->dim);
    return PCV_ERR_UNSUPPORTED;
  }
  if (rc != PCV_OK) return rc;
  ce_finalize_kernel<<<(unsigned)((M + 7) / 8), 256, 0, st>>>(
      part, p.n_split, M, t->dim, t->W, t->n_rows, t->row_offset, Q, targets, loss_rows, lse, dq, rec_out);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

int pcv_ce_fwd_bwd(const pcv_table *th, const float *Q, const int64_t *targets, int64_t M,
                   const pcv_ce_mask *mask, float *loss_rows, float *lse, float *dq,
                   void *workspace, size_t workspace_bytes, pcv_stream_t stream) {
  return ce_run(th, Q, targets, M, mask, loss_rows, lse, dq, nullptr, workspace, workspace_bytes, stream);
}

int pcv_ce_partials(const pcv_table *th, const float *Q, const int64_t *targets, int64_t M,
                    const pcv_ce_mask *mask, float *rec_out, void *workspace, size_t workspace_bytes,
                    pcv_stream_t stream) {
  PCV_CHECK_ARG(rec_out != nullptr, "rec_out is NULL");
  return ce_run(th, Q, targets, M, mask, nullptr, nullptr, nullptr, rec_out, workspace, workspace_bytes, stream);
}

int pcv_ce_vp_merge(const float *recs, int G, const float *W_full, int dim, const float *Q, const int64_t *targets,
                    int64_t M, float *loss_rows, float *lse, float *dq, pcv_stream_t stream) {
  PCV_CHECK_ARG(recs && W_full && Q && targets, "NULL pointer");
  PCV_CHECK_ARG(G >= 1 && M > 0 && dim >= 4 && dim <= 128, "bad shape");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  ce_vp_merge_kernel<<<(unsigned)((M + 127) / 128), 128, 0, (cudaStream_t)stream>>>(recs, G, M, dim, W_full, Q, targets,
                                                                                    loss_rows, lse, dq);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

}  // extern "C"
