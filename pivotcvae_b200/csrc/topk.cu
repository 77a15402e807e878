// topk.cu — exact streaming top-k over the catalog, and the opt-in no-repeat slate selection built on it.
//
// The reference has NO no-repeat logic (SURVEY F1: cvae.py:97-101 is an independent per-slot torch.max, duplicates
// inside a slate are allowed), so this is an extension, OFF by default; the rule it implements is the natural
// sequential one: slot l of a slate takes its best-scoring item (ties -> lowest index, SURVEY F2) that slots 0..l-1
// of the same slate have not taken.  Slot l excludes at most l items, so its answer is always among its own top-L:
//   1. the fast top-1 pass (score_select, tcgen05 engine) has already produced `items`;
//   2. nr_flag_kernel finds the slates that contain a duplicate (normally few) and compacts their rows;
//   3. topk_kernel re-scores ONLY those rows and keeps an exact top-L per row (same fp32 sequential-k FMA chain as
//      every other exact path, SURVEY F3);
//   4. nr_resolve_kernel walks each flagged slate slot by slot.
// The same kernel serves pcv_score_topk (torch.topk over the catalog, models/deterministic.py:119 in the reference).
// On a vocab-parallel catalog the global top-L of a row is the merge of the G shards' top-L lists: each rank runs
// steps 2-3 on its shard and writes its lists as pcv_pack_key keys by row (pcv_slate_no_repeat_partials); after an
// all-gather, nr_merge_kernel does step 4 over the G shard lists (pcv_slate_no_repeat_merge).
//
// topk_kernel layout: a CTA owns 8 warps x R query rows (registers) and one contiguous split of the catalog; tiles are
// staged with cp.async in the float4-SoA layout of score_select.cu; every lane keeps a sorted 16-entry (val, idx) list
// per row.  A lane visits its items in increasing index order, so a strict `>` against the list tail keeps the
// lowest-index entries among equal scores.  Warp merge = k rounds of (arg-max of the lane heads, pop the winner).
#include "pcv_common.cuh"

namespace pcv {

constexpr int TK_MAX = 16;            // list capacity = largest k (slate sizes are 5..10 in every config)
constexpr int TK_WARPS = 8;
constexpr int TK_THREADS = TK_WARPS * 32;
constexpr int TK_TILE_FLOATS = 8192;  // 32 KB per stage

template <int D>
struct TKCfg {
  static constexpr int R = (D <= 8) ? 2 : 1;            // rows per warp
  static constexpr int ROWS = TK_WARPS * R;             // rows per CTA
  static constexpr int TILE = (TK_TILE_FLOATS / D) < 128 ? 128 : (TK_TILE_FLOATS / D);
  static constexpr int C4 = D / 4;
  static constexpr size_t SMEM = 2ull * TILE * D * sizeof(float);
};

struct TKPlan {
  int rows_per_cta, row_tiles, n_split;
  int64_t items_per_split;
  size_t part_bytes;   // [n_split][M][TK_MAX] (val f32 + idx i32)
};

static int tk_plan(const Table *t, int64_t M, TKPlan *p) {
  int rows = 0, tile = 0;
  switch (t->dim) {
    case 4: rows = TKCfg<4>::ROWS; tile = TKCfg<4>::TILE; break;
    case 8: rows = TKCfg<8>::ROWS; tile = TKCfg<8>::TILE; break;
    case 16: rows = TKCfg<16>::ROWS; tile = TKCfg<16>::TILE; break;
    case 32: rows = TKCfg<32>::ROWS; tile = TKCfg<32>::TILE; break;
    case 64: rows = TKCfg<64>::ROWS; tile = TKCfg<64>::TILE; break;
    case 128: rows = TKCfg<128>::ROWS; tile = TKCfg<128>::TILE; break;
    default: return PCV_ERR_UNSUPPORTED;
  }
  p->rows_per_cta = rows;
  p->row_tiles = (int)((M + rows - 1) / rows);
  const int64_t n_tiles = (t->n_rows + tile - 1) / tile;
  // the number of rows that really need work is only known on the device (no-repeat: the flagged slates), so the
  // catalog is always cut in >= 8 splits: a handful of rows still spreads over the SMs
  int64_t ns = (4LL * t->sm_count + p->row_tiles - 1) / p->row_tiles;
  if (ns < 8) ns = 8;
  if (ns > 32) ns = 32;                       // the merge walks the splits with one lane each
  const int64_t max_split = (n_tiles + 3) / 4 > 0 ? (n_tiles + 3) / 4 : 1;
  if (ns > max_split) ns = max_split;
  const int64_t tps = (n_tiles + ns - 1) / ns;
  ns = (n_tiles + tps - 1) / tps;
  p->n_split = (int)ns;
  p->items_per_split = tps * tile;
  p->part_bytes = (size_t)ns * (size_t)M * TK_MAX * 8;
  return PCV_OK;
}

__device__ __forceinline__ void tk_cp_async16(void *smem, const void *gmem, bool valid) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(sz));
}

// rows: optional compact row list (row ids into Q) with its length on the device (n_rows_dev); NULL = rows 0..M-1.
template <int D>
__global__ void __launch_bounds__(TK_THREADS, (D <= 32 ? 2 : 1))
topk_kernel(const float *__restrict__ W, int64_t n_items, const float *__restrict__ Q, int64_t M,
            const int32_t *__restrict__ rows, const unsigned int *__restrict__ n_rows_dev, int64_t items_per_split,
            float *__restrict__ part_val, int32_t *__restrict__ part_idx) {
  using Cfg = TKCfg<D>;
  constexpr int R = Cfg::R, TILE = Cfg::TILE, C4 = Cfg::C4;
  const int64_t n_work = rows ? (int64_t)min((unsigned long long)M, (unsigned long long)*n_rows_dev) : M;
  const int64_t c0 = (int64_t)blockIdx.x * Cfg::ROWS;       // first compact row of this CTA
  if (c0 >= n_work) return;                                  // (whole CTA) nothing flagged here
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float4 *tile4 = reinterpret_cast<float4 *>(smem_raw);      // [2][C4][TILE]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t j_begin = (int64_t)blockIdx.y * items_per_split;
  const int64_t j_end = min(n_items, j_begin + items_per_split);
  const int n_tiles = (int)((j_end - j_begin + TILE - 1) / TILE);

  float q[R][D];
  float v[R][TK_MAX];
  int32_t ix[R][TK_MAX];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int64_t c = c0 + warp * R + r;
    const bool ok = c < n_work;
    const int64_t row = ok ? (rows ? (int64_t)rows[c] : c) : 0;
#pragma unroll
    for (int k = 0; k < C4; ++k) {
      const float4 t4 = ok ? __ldg(reinterpret_cast<const float4 *>(Q + row * D) + k) : make_float4(0.f, 0.f, 0.f, 0.f);
      q[r][4 * k + 0] = t4.x; q[r][4 * k + 1] = t4.y; q[r][4 * k + 2] = t4.z; q[r][4 * k + 3] = t4.w;
    }
#pragma unroll
    for (int e = 0; e < TK_MAX; ++e) { v[r][e] = -INFINITY; ix[r][e] = 0x7fffffff; }
  }

  auto load_tile = [&](int t, int buf) {
    const int64_t base = j_begin + (int64_t)t * TILE;
    float4 *dst = tile4 + (size_t)buf * C4 * TILE;
    const float4 *src = reinterpret_cast<const float4 *>(W + base * D);
#pragma unroll 4
    for (int f = threadIdx.x; f < TILE * C4; f += TK_THREADS) {
      const int item = f / C4, c = f % C4;
      const bool valid = (base + item) < j_end;
      tk_cp_async16(dst + c * TILE + item, valid ? (const void *)(src + f) : (const void *)W, valid);
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
#pragma unroll 2
    for (int i = lane; i < n_valid; i += 32) {
      float s[R];
#pragma unroll
      for (int r = 0; r < R; ++r) s[r] = 0.f;
#pragma unroll
      for (int c = 0; c < C4; ++c) {
        const float4 w4 = cur[c * TILE + i];
#pragma unroll
        for (int r = 0; r < R; ++r) {
          s[r] = fmaf(q[r][4 * c + 0], w4.x, s[r]);
          s[r] = fmaf(q[r][4 * c + 1], w4.y, s[r]);
          s[r] = fmaf(q[r][4 * c + 2], w4.z, s[r]);
          s[r] = fmaf(q[r][4 * c + 3], w4.w, s[r]);
        }
      }
      const int32_t j = (int32_t)(base + i);
#pragma unroll
      for (int r = 0; r < R; ++r) {
        if (s[r] > v[r][TK_MAX - 1]) {   // rare after the first few hundred items: replace the tail, bubble it up
          v[r][TK_MAX - 1] = s[r];
          ix[r][TK_MAX - 1] = j;
#pragma unroll
          for (int e = TK_MAX - 1; e > 0; --e) {
            if (v[r][e] > v[r][e - 1]) {   // strict: an equal score with a larger index stays below
              const float tv = v[r][e]; v[r][e] = v[r][e - 1]; v[r][e - 1] = tv;
              const int32_t ti = ix[r][e]; ix[r][e] = ix[r][e - 1]; ix[r][e - 1] = ti;
            }
          }
        }
      }
    }
    __syncthreads();
  }

  // warp merge: TK_MAX rounds of (best lane head, ties -> lowest index), the winning lane pops its head
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int64_t c = c0 + warp * R + r;
    for (int round = 0; round < TK_MAX; ++round) {
      float bv = v[r][0];
      int32_t bi = ix[r][0];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int32_t oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
      }
      if (bi == ix[r][0] && bi != 0x7fffffff) {   // item ids are unique across lanes: exactly one lane pops
#pragma unroll
        for (int e = 0; e < TK_MAX - 1; ++e) { v[r][e] = v[r][e + 1]; ix[r][e] = ix[r][e + 1]; }
        v[r][TK_MAX - 1] = -INFINITY;
        ix[r][TK_MAX - 1] = 0x7fffffff;
      }
      if (lane == 0 && c < n_work) {
        const size_t o = (((size_t)blockIdx.y * M + c) * TK_MAX) + round;
        part_val[o] = bv;
        part_idx[o] = bi;
      }
    }
  }
}

// The sorted lists tk_merge_row reads, as pcv_pack_key keys with global indices.
// topk_kernel's per-split partials: (val, local idx), empty entries hold idx 0x7fffffff.
struct TkSplitLists {
  const float *val;
  const int32_t *idx;
  int64_t row_offset;
  __device__ __forceinline__ long long operator()(size_t o) const {
    const int32_t i = idx[o];
    return i == 0x7fffffff ? PCV_KEY_NONE : pcv_pack_key(val[o], (int64_t)i + row_offset);
  }
};
// Keys already packed (the shard lists of pcv_slate_no_repeat_partials).
struct TkKeyLists {
  const long long *keys;
  __device__ __forceinline__ long long operator()(size_t o) const { return keys[o]; }
};

// k-way merge of sorted lists of `len` entries, one lane per list: list g of row `row` starts at
// g * list_stride + row * len.  The lists hold disjoint items (catalog splits or shards), so keys are unique and
// exactly one lane pops per round.  Emits the e-th best key (PCV_KEY_NONE past the end) lane-uniformly.
template <class Lists, class F>
__device__ __forceinline__ void tk_merge_row(const Lists &lists, int n_lists, size_t list_stride, int64_t row, int len,
                                             int k, F &&emit) {
  const int lane = threadIdx.x & 31;
  int cur = 0;
  for (int e = 0; e < k; ++e) {
    const long long head = (lane < n_lists && cur < len) ? lists((size_t)lane * list_stride + (size_t)row * len + cur)
                                                         : PCV_KEY_NONE;
    long long best = head;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const long long other = __shfl_xor_sync(0xffffffffu, best, o);
      best = other > best ? other : best;
    }
    if (best == head && best != PCV_KEY_NONE) ++cur;
    emit(e, best);
  }
}

__global__ void topk_finalize_kernel(const float *__restrict__ part_val, const int32_t *__restrict__ part_idx, int n_split,
                                     int64_t M, int k, int64_t row_offset, int64_t *__restrict__ out_idx,
                                     float *__restrict__ out_val) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const int lane = threadIdx.x & 31;
  tk_merge_row(TkSplitLists{part_val, part_idx, row_offset}, n_split, (size_t)M * TK_MAX, row, TK_MAX, k,
               [&](int e, long long key) {
    if (lane == 0) {
      int64_t ix;
      const float v = pcv_unpack_key(key, ix);
      out_idx[row * k + e] = key == PCV_KEY_NONE ? (int64_t)-1 : ix;   // -1: fewer than k items
      if (out_val) out_val[row * k + e] = key == PCV_KEY_NONE ? -INFINITY : v;
    }
  });
}

// ---- no-repeat
// slate b holds a duplicate among its picks
__device__ __forceinline__ bool nr_has_dup(const int64_t *__restrict__ items, int64_t b, int L) {
  for (int l = 1; l < L; ++l)
    for (int m = 0; m < l; ++m)
      if (items[b * L + l] == items[b * L + m]) return true;
  return false;
}

// flag the slates that hold a duplicate and list their rows (slot order kept)
__global__ void nr_flag_kernel(const int64_t *__restrict__ items, int64_t B, int L, unsigned int *__restrict__ n_rows_dev,
                               int32_t *__restrict__ rows) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  if (nr_has_dup(items, b, L)) {
    const unsigned int pos = atomicAdd(n_rows_dev, (unsigned int)L);
    for (int l = 0; l < L; ++l) rows[pos + l] = (int32_t)(b * L + l);
  }
}

// Slot-by-slot resolve of one slate by one warp: merge_row(l, emit) streams slot l's candidates best first as keys;
// slot l takes the first whose item slots 0..l-1 have not taken, and take(l, item, val) stores it.
template <class MergeRow, class Take>
__device__ __forceinline__ void nr_resolve_slate(int L, MergeRow &&merge_row, Take &&take) {
  int64_t taken[TK_MAX];
#pragma unroll
  for (int e = 0; e < TK_MAX; ++e) taken[e] = -1;
  for (int l = 0; l < L; ++l) {
    bool done = false;
    merge_row(l, [&](int e, long long key) {
      if (done || key == PCV_KEY_NONE) return;
      int64_t item;
      const float v = pcv_unpack_key(key, item);
      bool used = false;
#pragma unroll
      for (int m = 0; m < TK_MAX; ++m) used |= (m < l && taken[m] == item);
      if (!used) {
        done = true;
#pragma unroll
        for (int m = 0; m < TK_MAX; ++m) if (m == l) taken[m] = item;
        take(l, item, v);
      }
    });
  }
}

// one warp per flagged slate: the top-L lists of its rows come from the catalog splits of this table
__global__ void nr_resolve_kernel(const float *__restrict__ part_val, const int32_t *__restrict__ part_idx, int n_split,
                                  int64_t M, int L, int64_t row_offset, const int32_t *__restrict__ rows,
                                  unsigned int *__restrict__ n_rows_dev, int64_t *__restrict__ items,
                                  float *__restrict__ vals) {
  const int64_t s = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);   // flagged slate
  const int64_t n_work = min((unsigned long long)M, (unsigned long long)*n_rows_dev);
  if (s * L >= n_work) return;
  const int lane = threadIdx.x & 31;
  const TkSplitLists lists{part_val, part_idx, row_offset};
  nr_resolve_slate(L, [&](int l, auto &&emit) { tk_merge_row(lists, n_split, (size_t)M * TK_MAX, s * L + l, TK_MAX, L, emit); },
                   [&](int l, int64_t item, float v) {
    if (lane == 0) {
      items[rows[s * L + l]] = item;
      if (vals) vals[rows[s * L + l]] = v;
    }
  });
}

__global__ void nr_reset_kernel(unsigned int *n_rows_dev) { *n_rows_dev = 0u; }

// ---- no-repeat over a vocab-parallel catalog: shard partials + merge of the G shards' lists
// counter reset + every key PCV_KEY_NONE (duplicate-free slates, and entries past the end of a small shard)
__global__ void nr_partials_init_kernel(unsigned int *__restrict__ n_rows_dev, long long *__restrict__ keys, int64_t n) {
  const int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i0 == 0) *n_rows_dev = 0u;
  for (int64_t i = i0; i < n; i += (int64_t)gridDim.x * blockDim.x) keys[i] = PCV_KEY_NONE;
}

// one warp per compact (flagged) row: this shard's top-L, scattered to the row's own place so that the lists of all
// ranks line up (the compact order comes from atomics and differs between ranks)
__global__ void nr_partials_kernel(const float *__restrict__ part_val, const int32_t *__restrict__ part_idx, int n_split,
                                   int64_t M, int L, int64_t row_offset, const int32_t *__restrict__ rows,
                                   const unsigned int *__restrict__ n_rows_dev, long long *__restrict__ keys) {
  const int64_t c = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_work = min((unsigned long long)M, (unsigned long long)*n_rows_dev);
  if (c >= n_work) return;
  const int lane = threadIdx.x & 31;
  const int64_t row = rows[c];
  tk_merge_row(TkSplitLists{part_val, part_idx, row_offset}, n_split, (size_t)M * TK_MAX, c, TK_MAX, L,
               [&](int e, long long key) {
    if (lane == 0) keys[row * L + e] = key;
  });
}

// one warp per slate: re-detects the duplicate from the (replicated) picks, so no compaction and the same result
// on every rank; the top-L lists of its rows come from the G shards (one lane each, shards in index order)
__global__ void nr_merge_kernel(const long long *__restrict__ keys, int G, int64_t B, int L, int64_t *__restrict__ items,
                                float *__restrict__ vals) {
  const int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= B || !nr_has_dup(items, b, L)) return;
  const int lane = threadIdx.x & 31;
  const size_t M = (size_t)B * L;
  __syncwarp();   // every lane has read the picks before lane 0 rewrites them
  nr_resolve_slate(L, [&](int l, auto &&emit) { tk_merge_row(TkKeyLists{keys}, G, M * L, b * L + l, L, L, emit); },
                   [&](int l, int64_t item, float v) {
    if (lane == 0) {
      items[b * L + l] = item;
      if (vals) vals[b * L + l] = v;
    }
  });
}

template <int D>
static int launch_topk(const Table *t, const TKPlan &p, const float *Q, int64_t M, const int32_t *rows,
                       const unsigned int *n_rows_dev, float *pv, int32_t *pi, cudaStream_t st) {
  using Cfg = TKCfg<D>;
  auto kern = topk_kernel<D>;
  static bool attr_set[64] = {false};
  if (!attr_set[t->device & 63]) {
    PCV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM));
    attr_set[t->device & 63] = true;
  }
  dim3 grid((unsigned)p.row_tiles, (unsigned)p.n_split);
  kern<<<grid, TK_THREADS, Cfg::SMEM, st>>>(t->W, t->n_rows, Q, M, rows, n_rows_dev, p.items_per_split, pv, pi);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

static int dispatch_topk(const Table *t, const TKPlan &p, const float *Q, int64_t M, const int32_t *rows,
                         const unsigned int *n_rows_dev, float *pv, int32_t *pi, cudaStream_t st) {
  switch (t->dim) {
    case 4: return launch_topk<4>(t, p, Q, M, rows, n_rows_dev, pv, pi, st);
    case 8: return launch_topk<8>(t, p, Q, M, rows, n_rows_dev, pv, pi, st);
    case 16: return launch_topk<16>(t, p, Q, M, rows, n_rows_dev, pv, pi, st);
    case 32: return launch_topk<32>(t, p, Q, M, rows, n_rows_dev, pv, pi, st);
    case 64: return launch_topk<64>(t, p, Q, M, rows, n_rows_dev, pv, pi, st);
    case 128: return launch_topk<128>(t, p, Q, M, rows, n_rows_dev, pv, pi, st);
  }
  set_error("score_topk: dim %d unsupported (use 4, 8, 16, 32, 64 or 128)", t->dim);
  return PCV_ERR_UNSUPPORTED;
}

}  // namespace pcv

using namespace pcv;

extern "C" {

int pcv_score_topk_workspace_bytes(const pcv_table *th, int64_t M, size_t *bytes_host) {
  PCV_CHECK_ARG(th && bytes_host, "NULL pointer");
  PCV_CHECK_ARG(M > 0, "M must be > 0");
  const Table *t = reinterpret_cast<const Table *>(th);
  TKPlan p;
  if (tk_plan(t, M, &p) != PCV_OK) {
    set_error("score_topk: dim %d unsupported", t->dim);
    return PCV_ERR_UNSUPPORTED;
  }
  // 256 (device counter) + compact row list + partial lists
  *bytes_host = (256 + (((size_t)M * 4 + 255) & ~(size_t)255) + p.part_bytes + 255) & ~(size_t)255;
  return PCV_OK;
}

int pcv_score_topk(const pcv_table *th, const float *Q, int64_t M, int k, int64_t *out_idx, float *out_val,
                   void *workspace, size_t workspace_bytes, pcv_stream_t stream) {
  PCV_CHECK_ARG(th && Q && out_idx, "NULL pointer");
  PCV_CHECK_ARG(M > 0, "M must be > 0");
  PCV_CHECK_ARG(k >= 1 && k <= TK_MAX, "k must be in [1, 16]");
  const Table *t = reinterpret_cast<const Table *>(th);
  PCV_CHECK_ARG(t->n_rows < 0x7fffffffLL, "shard larger than 2^31-1 rows");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  size_t need = 0;
  rc = pcv_score_topk_workspace_bytes(th, M, &need);
  if (rc != PCV_OK) return rc;
  if (workspace == nullptr || workspace_bytes < need) {
    set_error("score_topk: workspace too small (%zu < %zu)", workspace_bytes, need);
    return PCV_ERR_WORKSPACE;
  }
  TKPlan p;
  tk_plan(t, M, &p);
  cudaStream_t st = (cudaStream_t)stream;
  char *base = static_cast<char *>(workspace) + 256 + (((size_t)M * 4 + 255) & ~(size_t)255);
  float *pv = reinterpret_cast<float *>(base);
  int32_t *pi = reinterpret_cast<int32_t *>(pv + (size_t)p.n_split * M * TK_MAX);
  rc = dispatch_topk(t, p, Q, M, nullptr, nullptr, pv, pi, st);
  if (rc != PCV_OK) return rc;
  topk_finalize_kernel<<<(unsigned)((M + 7) / 8), 256, 0, st>>>(pv, pi, p.n_split, M, k, t->row_offset, out_idx, out_val);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

int pcv_slate_no_repeat(const pcv_table *th, const float *Q, int64_t B, int L, int64_t *items, float *vals,
                        void *workspace, size_t workspace_bytes, pcv_stream_t stream) {
  PCV_CHECK_ARG(th && Q && items, "NULL pointer");
  PCV_CHECK_ARG(B > 0, "B must be > 0");
  PCV_CHECK_ARG(L >= 1 && L <= TK_MAX, "slate size must be in [1, 16]");
  const Table *t = reinterpret_cast<const Table *>(th);
  PCV_CHECK_ARG(t->row_offset == 0, "no-repeat selection needs the whole catalog (row_offset 0)");
  PCV_CHECK_ARG(t->n_rows >= L, "catalog smaller than the slate");
  PCV_CHECK_ARG(t->n_rows < 0x7fffffffLL && B * L < 0x7fffffffLL, "problem too large for 32-bit row ids");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  const int64_t M = B * L;
  size_t need = 0;
  rc = pcv_score_topk_workspace_bytes(th, M, &need);
  if (rc != PCV_OK) return rc;
  if (workspace == nullptr || workspace_bytes < need) {
    set_error("slate_no_repeat: workspace too small (%zu < %zu)", workspace_bytes, need);
    return PCV_ERR_WORKSPACE;
  }
  if (L == 1) return PCV_OK;
  TKPlan p;
  tk_plan(t, M, &p);
  cudaStream_t st = (cudaStream_t)stream;
  unsigned int *n_rows_dev = static_cast<unsigned int *>(workspace);
  int32_t *rows = reinterpret_cast<int32_t *>(static_cast<char *>(workspace) + 256);
  char *base = static_cast<char *>(workspace) + 256 + (((size_t)M * 4 + 255) & ~(size_t)255);
  float *pv = reinterpret_cast<float *>(base);
  int32_t *pi = reinterpret_cast<int32_t *>(pv + (size_t)p.n_split * M * TK_MAX);
  nr_reset_kernel<<<1, 1, 0, st>>>(n_rows_dev);
  PCV_LAUNCH_CHECK();
  nr_flag_kernel<<<(unsigned)((B + 255) / 256), 256, 0, st>>>(items, B, L, n_rows_dev, rows);
  PCV_LAUNCH_CHECK();
  rc = dispatch_topk(t, p, Q, M, rows, n_rows_dev, pv, pi, st);
  if (rc != PCV_OK) return rc;
  nr_resolve_kernel<<<(unsigned)((B + 7) / 8), 256, 0, st>>>(pv, pi, p.n_split, M, L, t->row_offset, rows, n_rows_dev,
                                                           items, vals);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

int pcv_slate_no_repeat_partials(const pcv_table *th, const float *Q, int64_t B, int L, const int64_t *items,
                                 int64_t *keys, void *workspace, size_t workspace_bytes, pcv_stream_t stream) {
  PCV_CHECK_ARG(th && Q && items && keys, "NULL pointer");
  PCV_CHECK_ARG(B > 0, "B must be > 0");
  PCV_CHECK_ARG(L >= 1 && L <= TK_MAX, "slate size must be in [1, 16]");
  const Table *t = reinterpret_cast<const Table *>(th);
  PCV_CHECK_ARG(t->n_rows < 0x7fffffffLL && B * L < 0x7fffffffLL, "problem too large for 32-bit row ids");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  const int64_t M = B * L;
  size_t need = 0;
  rc = pcv_score_topk_workspace_bytes(th, M, &need);
  if (rc != PCV_OK) return rc;
  if (workspace == nullptr || workspace_bytes < need) {
    set_error("slate_no_repeat_partials: workspace too small (%zu < %zu)", workspace_bytes, need);
    return PCV_ERR_WORKSPACE;
  }
  TKPlan p;
  tk_plan(t, M, &p);
  cudaStream_t st = (cudaStream_t)stream;
  unsigned int *n_rows_dev = static_cast<unsigned int *>(workspace);
  int32_t *rows = reinterpret_cast<int32_t *>(static_cast<char *>(workspace) + 256);
  char *base = static_cast<char *>(workspace) + 256 + (((size_t)M * 4 + 255) & ~(size_t)255);
  float *pv = reinterpret_cast<float *>(base);
  int32_t *pi = reinterpret_cast<int32_t *>(pv + (size_t)p.n_split * M * TK_MAX);
  long long *k = reinterpret_cast<long long *>(keys);
  const int64_t n_keys = M * L;
  const int64_t init_blocks = (n_keys + 255) / 256 < 1024 ? (n_keys + 255) / 256 : 1024;
  nr_partials_init_kernel<<<(unsigned)init_blocks, 256, 0, st>>>(n_rows_dev, k, n_keys);
  PCV_LAUNCH_CHECK();
  if (L == 1) return PCV_OK;   // a one-item slate never repeats
  nr_flag_kernel<<<(unsigned)((B + 255) / 256), 256, 0, st>>>(items, B, L, n_rows_dev, rows);
  PCV_LAUNCH_CHECK();
  rc = dispatch_topk(t, p, Q, M, rows, n_rows_dev, pv, pi, st);
  if (rc != PCV_OK) return rc;
  nr_partials_kernel<<<(unsigned)((M + 7) / 8), 256, 0, st>>>(pv, pi, p.n_split, M, L, t->row_offset, rows, n_rows_dev, k);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

int pcv_slate_no_repeat_merge(const int64_t *keys, int G, int64_t B, int L, int64_t *items, float *vals,
                              pcv_stream_t stream) {
  PCV_CHECK_ARG(keys && items, "NULL pointer");
  PCV_CHECK_ARG(B > 0, "B must be > 0");
  PCV_CHECK_ARG(L >= 1 && L <= TK_MAX, "slate size must be in [1, 16]");
  PCV_CHECK_ARG(G >= 1 && G <= 32, "G must be in [1, 32] (one lane per shard)");
  PCV_CHECK_ARG(B * L < 0x7fffffffLL, "problem too large for 32-bit row ids");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  nr_merge_kernel<<<(unsigned)((B + 7) / 8), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const long long *>(keys),
                                                                             G, B, L, items, vals);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

}  // extern "C"
