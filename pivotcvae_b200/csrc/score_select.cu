// score_select.cu — fused full-catalog scoring + selection, exact-fp32 engine.
//
// Replaces (reference file:line)
//   cvae.py:97-101        get_recommended_item: mm((B*L,D),(D,N)) -> torch.max(p,1)
//   pivotcvae.py:191      pick_pivot (greedy):  mm((N,D),(D,B)).max(0)[1]
//   pivotcvae.py:349-351  pick_pivot (sampled): Categorical(sigmoid(mm)).sample()
//   pivotcvae.py:274      forward(): p = mm(prox_emb, table.t())   (pcv_score_logits)
//
// Arithmetic contract (SURVEY F2/F3): score = fma(q[D-1],w[D-1], ... fma(q[0],w[0],0)),
// k ascending; winner = largest score, equal scores -> lowest item index.  The
// (M x N) logit matrix never reaches HBM (except through pcv_score_logits).
//
// Layout: a CTA owns ROWS = 8 warps x R query rows (held in registers) and one
// contiguous split of the catalog; catalog tiles of TILE items are staged into
// shared memory with cp.async (double buffered) in a float4-SoA layout
// ([chunk][item], conflict-free for lane<->item), and every warp scores the whole
// tile against its own R rows.  Per-split partial winners go to the workspace and
// a second tiny kernel merges the splits.
#include "pcv_common.cuh"

namespace pcv {

constexpr int SS_WARPS = 8;
constexpr int SS_THREADS = SS_WARPS * 32;
constexpr int SS_TILE_FLOATS = 8192;  // 32 KB per stage

enum { SS_GREEDY = 0, SS_EXPRACE_NOISE = 1, SS_LOGITS = 3 };

template <int D>
struct SSCfg {
  static constexpr int R = (D <= 8) ? 8 : (D <= 64 ? 64 / D : 1);  // rows per warp
  static constexpr int ROWS = SS_WARPS * R;                        // rows per CTA
  static constexpr int TILE = (SS_TILE_FLOATS / D) < 128 ? 128 : (SS_TILE_FLOATS / D);
  static constexpr int C4 = D / 4;                                 // float4 chunks per item
  static constexpr size_t SMEM = 2ull * TILE * D * sizeof(float);
};

struct SSPlan {
  int rows_per_cta, tile;
  int row_tiles, n_split;
  int64_t items_per_split;  // multiple of tile
  size_t ws_bytes;
};

static int rows_per_cta_for(int D) {
  switch (D) {
    case 4: return SSCfg<4>::ROWS;
    case 8: return SSCfg<8>::ROWS;
    case 16: return SSCfg<16>::ROWS;
    case 32: return SSCfg<32>::ROWS;
    case 64: return SSCfg<64>::ROWS;
    case 128: return SSCfg<128>::ROWS;
  }
  return 0;
}
static int tile_for(int D) {
  int t = SS_TILE_FLOATS / D;
  return t < 128 ? 128 : t;
}

// The partial winners sit behind the head of the workspace that the tcgen05 engine needs zero on entry (its overflow
// counter and per-row overflow winners: score_select_tc.cu), so that the engines can share one workspace in any order.
static size_t ss_ws_head(int64_t M) { return 256 + (((size_t)M * 8 + 255) & ~(size_t)255); }

static int make_plan(const Table *t, int64_t M, SSPlan *p) {
  p->rows_per_cta = rows_per_cta_for(t->dim);
  if (p->rows_per_cta == 0) return PCV_ERR_UNSUPPORTED;
  p->tile = tile_for(t->dim);
  p->row_tiles = (int)((M + p->rows_per_cta - 1) / p->rows_per_cta);
  int64_t n_tiles = (t->n_rows + p->tile - 1) / p->tile;
  // aim for >= 4 CTAs per SM in flight (2 resident + 2 queued) so the tail is short
  int64_t want = (4LL * t->sm_count + p->row_tiles - 1) / p->row_tiles;
  int64_t max_split = (n_tiles + 3) / 4;  // keep >= 4 tiles per split
  if (max_split < 1) max_split = 1;
  int64_t ns = want < 1 ? 1 : (want > max_split ? max_split : want);
  int64_t tiles_per_split = (n_tiles + ns - 1) / ns;
  ns = (n_tiles + tiles_per_split - 1) / tiles_per_split;
  p->n_split = (int)ns;
  p->items_per_split = tiles_per_split * p->tile;
  p->ws_bytes = ss_ws_head(M) + (size_t)ns * (size_t)M * (sizeof(float) + sizeof(int32_t));
  return PCV_OK;
}

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem, bool valid) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  int sz = valid ? 16 : 0;  // src-size 0 -> zero fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

template <int D, int MODE>
__global__ void __launch_bounds__(SS_THREADS, (D <= 32 ? 2 : 1))
score_select_kernel(const float *__restrict__ W, int64_t n_rows,
                    const float *__restrict__ Q, int64_t M, int64_t items_per_split,
                    const float *__restrict__ noise, float *__restrict__ part_val,
                    int32_t *__restrict__ part_idx, float *__restrict__ logits_out) {
  using Cfg = SSCfg<D>;
  constexpr int R = Cfg::R, TILE = Cfg::TILE, C4 = Cfg::C4;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float4 *tile4 = reinterpret_cast<float4 *>(smem_raw);  // [2][C4][TILE]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row0 = (int64_t)blockIdx.x * Cfg::ROWS + (int64_t)warp * R;
  const int64_t j_begin = (int64_t)blockIdx.y * items_per_split;
  const int64_t j_end = min(n_rows, j_begin + items_per_split);
  const int n_tiles = (int)((j_end - j_begin + TILE - 1) / TILE);

  // query rows -> registers (rows beyond M read as zero and are never written)
  float q[R][D];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const bool ok = (row0 + r) < M;
#pragma unroll
    for (int c = 0; c < C4; ++c) {
      float4 v = ok ? __ldg(reinterpret_cast<const float4 *>(Q + (row0 + r) * D) + c)
                    : make_float4(0.f, 0.f, 0.f, 0.f);
      q[r][4 * c + 0] = v.x; q[r][4 * c + 1] = v.y; q[r][4 * c + 2] = v.z; q[r][4 * c + 3] = v.w;
    }
  }
  float best[R];
  int32_t bidx[R];
#pragma unroll
  for (int r = 0; r < R; ++r) { best[r] = -INFINITY; bidx[r] = 0x7fffffff; }

  auto load_tile = [&](int t, int buf) {
    const int64_t base = j_begin + (int64_t)t * TILE;
    float4 *dst = tile4 + (size_t)buf * C4 * TILE;
    const float4 *src = reinterpret_cast<const float4 *>(W + base * D);
#pragma unroll 4
    for (int f = threadIdx.x; f < TILE * C4; f += SS_THREADS) {
      int item = f / C4, c = f % C4;
      bool valid = (base + item) < j_end;
      cp_async16(dst + c * TILE + item, valid ? (const void *)(src + f) : (const void *)W, valid);
    }
    cp_async_commit();
  };

  if (n_tiles > 0) load_tile(0, 0);
  for (int t = 0; t < n_tiles; ++t) {
    if (t + 1 < n_tiles) {
      load_tile(t + 1, (t + 1) & 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
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
        const float4 v = cur[c * TILE + i];
#pragma unroll
        for (int r = 0; r < R; ++r) {
          s[r] = fmaf(q[r][4 * c + 0], v.x, s[r]);
          s[r] = fmaf(q[r][4 * c + 1], v.y, s[r]);
          s[r] = fmaf(q[r][4 * c + 2], v.z, s[r]);
          s[r] = fmaf(q[r][4 * c + 3], v.w, s[r]);
        }
      }
      const int32_t j = (int32_t)(base + i);
#pragma unroll
      for (int r = 0; r < R; ++r) {
        if (MODE == SS_LOGITS) {
          if (row0 + r < M) logits_out[(row0 + r) * n_rows + j] = s[r];
        } else {
          float key = s[r];
          if (MODE == SS_EXPRACE_NOISE) {
            // race time T = E * (1 + exp(-s)) = E / sigmoid(s); winner = min T.
            float e = (row0 + r < M) ? __ldg(noise + (row0 + r) * n_rows + j) : 1.f;
            key = -(e * (1.0f + pcv_expf(-s[r])));
          }
          if (key > best[r]) { best[r] = key; bidx[r] = j; }
        }
      }
    }
    __syncthreads();
  }

  if constexpr (MODE != SS_LOGITS) {
    // lanes saw disjoint, increasing item sets: merge with lowest-index ties
#pragma unroll
    for (int r = 0; r < R; ++r) {
      float v = best[r];
      int32_t ix = bidx[r];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        float ov = __shfl_xor_sync(0xffffffffu, v, o);
        int32_t oi = __shfl_xor_sync(0xffffffffu, ix, o);
        if (ov > v || (ov == v && oi < ix)) { v = ov; ix = oi; }
      }
      if (lane == 0 && row0 + r < M) {
        part_val[(int64_t)blockIdx.y * M + row0 + r] = v;
        part_idx[(int64_t)blockIdx.y * M + row0 + r] = ix;
      }
    }
  }
}

// Merge the per-split partial winners (splits are in ascending item order).
__global__ void select_finalize_kernel(const float *__restrict__ part_val,
                                       const int32_t *__restrict__ part_idx, int n_split,
                                       int64_t M, int64_t row_offset,
                                       int64_t *__restrict__ out_idx, float *__restrict__ out_val) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  float v = part_val[i];
  int32_t ix = part_idx[i];
  for (int s = 1; s < n_split; ++s) {
    float ov = part_val[(int64_t)s * M + i];
    int32_t oi = part_idx[(int64_t)s * M + i];
    if (ov > v || (ov == v && oi < ix)) { v = ov; ix = oi; }
  }
  if (ix == 0x7fffffff) ix = 0;   // no score above -inf (NaN never wins): the first index, value -inf (pcv_b200.h)
  out_idx[i] = (int64_t)ix + row_offset;
  if (out_val) out_val[i] = v;
}

// Vocab-parallel exchange as ONE all-reduce(MAX) on int64 keys (pcv_pack_key): the signed maximum over the shards
// is the largest value, equal values -> lowest global index (the reference's tie rule, SURVEY F2).
__global__ void vp_pack_keys_kernel(const float *__restrict__ vals, const int64_t *__restrict__ idx, int64_t M,
                                    long long *__restrict__ keys) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  keys[i] = pcv_pack_key(vals[i], idx[i]);
}

__global__ void vp_unpack_keys_kernel(const long long *__restrict__ keys, int64_t M, int64_t *__restrict__ out_idx,
                                      float *__restrict__ out_val) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  int64_t ix;
  const float v = pcv_unpack_key(keys[i], ix);
  out_idx[i] = ix;
  if (out_val) out_val[i] = v;
}

template <int D, int MODE>
static int launch_ss(const Table *t, const SSPlan &p, const float *Q, int64_t M, const float *noise,
                     float *pv, int32_t *pi, float *logits, cudaStream_t st) {
  using Cfg = SSCfg<D>;
  auto kern = score_select_kernel<D, MODE>;
  static bool attr_set[64] = {false};  // per instantiation, per device
  if (!attr_set[t->device & 63]) {
    PCV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM));
    attr_set[t->device & 63] = true;
  }
  dim3 grid((unsigned)p.row_tiles, (unsigned)p.n_split);
  kern<<<grid, SS_THREADS, Cfg::SMEM, st>>>(t->W, t->n_rows, Q, M, p.items_per_split, noise, pv, pi, logits);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

template <int MODE>
static int dispatch_dim(const Table *t, const SSPlan &p, const float *Q, int64_t M, const float *noise,
                        float *pv, int32_t *pi, float *logits, cudaStream_t st) {
  switch (t->dim) {
    case 4: return launch_ss<4, MODE>(t, p, Q, M, noise, pv, pi, logits, st);
    case 8: return launch_ss<8, MODE>(t, p, Q, M, noise, pv, pi, logits, st);
    case 16: return launch_ss<16, MODE>(t, p, Q, M, noise, pv, pi, logits, st);
    case 32: return launch_ss<32, MODE>(t, p, Q, M, noise, pv, pi, logits, st);
    case 64: return launch_ss<64, MODE>(t, p, Q, M, noise, pv, pi, logits, st);
    case 128: return launch_ss<128, MODE>(t, p, Q, M, noise, pv, pi, logits, st);
  }
  set_error("score_select: dim %d unsupported (use 4, 8, 16, 32, 64 or 128)", t->dim);
  return PCV_ERR_UNSUPPORTED;
}

void launch_select_finalize(const float *pv, const int32_t *pi, int n_parts, int64_t M, int64_t row_offset,
                            int64_t *out_idx, float *out_val, cudaStream_t st) {
  const int threads = 256;
  select_finalize_kernel<<<(unsigned)((M + threads - 1) / threads), threads, 0, st>>>(pv, pi, n_parts, M, row_offset,
                                                                                       out_idx, out_val);
}

// tcgen05 engine (score_select_tc.cu)
int score_select_tc(const Table *t, const float *Q, int64_t M, int64_t *out_idx, float *out_val,
                    void *ws, size_t ws_bytes, cudaStream_t st, int f16);
size_t score_select_tc_workspace(const Table *t, int64_t M);
bool score_select_tc_supported(const Table *t);
bool score_select_tc_f16_supported(const Table *t);

}  // namespace pcv

using namespace pcv;

extern "C" {

int pcv_score_select_workspace_bytes(const pcv_table *th, int64_t M, size_t *bytes_host) {
  PCV_CHECK_ARG(th && bytes_host, "NULL pointer");
  PCV_CHECK_ARG(M > 0, "M must be > 0");
  const Table *t = reinterpret_cast<const Table *>(th);
  SSPlan p;
  if (make_plan(t, M, &p) != PCV_OK) {
    set_error("score_select: dim %d unsupported", t->dim);
    return PCV_ERR_UNSUPPORTED;
  }
  size_t b = p.ws_bytes;
  size_t tc = score_select_tc_workspace(t, M);
  if (tc > b) b = tc;
  *bytes_host = (b + 255) & ~(size_t)255;
  return PCV_OK;
}

int pcv_score_select(const pcv_table *th, const float *Q, int64_t M,
                     const pcv_select_opts *opts, int64_t *out_idx, float *out_val,
                     void *workspace, size_t workspace_bytes, pcv_stream_t stream) {
  PCV_CHECK_ARG(th && Q && opts && out_idx, "NULL pointer");
  PCV_CHECK_ARG(M > 0, "M must be > 0");
  PCV_CHECK_ARG(opts->mode == PCV_SELECT_GREEDY || opts->mode == PCV_SELECT_EXPRACE, "bad mode");
  PCV_CHECK_ARG(opts->mode != PCV_SELECT_EXPRACE || opts->noise,
                "exprace needs the [M, n_rows] Exp(1) noise (sampled pivots without it: pcv_sigmoid_categorical)");
  const Table *t = reinterpret_cast<const Table *>(th);
  if (opts->no_repeat != 0) {
    // opt-in extension (the reference has no mask, SURVEY F1): top-1 pass on the head of the workspace, then the
    // duplicate-holding slates are re-selected sequentially by pcv_slate_no_repeat on the tail of it
    const int Ls = opts->no_repeat;
    PCV_CHECK_ARG(Ls >= 1 && Ls <= 16, "no_repeat must be the slate size (1..16)");
    PCV_CHECK_ARG(opts->mode == PCV_SELECT_GREEDY, "no_repeat needs greedy mode");
    PCV_CHECK_ARG(M % Ls == 0, "no_repeat: M must be a multiple of the slate size");
    size_t head = 0, tail = 0;
    int rc0 = pcv_score_select_workspace_bytes(th, M, &head);
    if (rc0 == PCV_OK) rc0 = pcv_score_topk_workspace_bytes(th, M, &tail);
    if (rc0 != PCV_OK) return rc0;
    if (workspace == nullptr || workspace_bytes < head + tail) {
      set_error("score_select(no_repeat): workspace too small (%zu < %zu + %zu)", workspace_bytes, head, tail);
      return PCV_ERR_WORKSPACE;
    }
    pcv_select_opts o = *opts;
    o.no_repeat = 0;
    rc0 = pcv_score_select(th, Q, M, &o, out_idx, out_val, workspace, head, stream);
    if (rc0 != PCV_OK) return rc0;
    return pcv_slate_no_repeat(th, Q, M / Ls, Ls, out_idx, out_val, static_cast<char *>(workspace) + head, tail, stream);
  }
  PCV_CHECK_ARG(t->n_rows < 0x7fffffffLL, "shard larger than 2^31-1 rows");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;

  int engine = opts->engine;
  if (engine == PCV_ENGINE_AUTO)  // tensor cores whenever the shape allows and the catalog is not tiny; dim 8: the f16 filter
    engine = (opts->mode == PCV_SELECT_GREEDY && score_select_tc_supported(t) && t->n_rows >= 2048)
                 ? (score_select_tc_f16_supported(t) ? PCV_ENGINE_TCGEN05_F16 : PCV_ENGINE_TCGEN05) : PCV_ENGINE_SIMT;
  if (engine == PCV_ENGINE_TCGEN05 || engine == PCV_ENGINE_TCGEN05_F16) {
    if (opts->mode != PCV_SELECT_GREEDY || !score_select_tc_supported(t)) {
      set_error("score_select: tcgen05 engine needs greedy mode and dim 8, 16, 32, 64 or 128 (dim %d, mode %d)", t->dim, opts->mode);
      return PCV_ERR_UNSUPPORTED;
    }
    return score_select_tc(t, Q, M, out_idx, out_val, workspace, workspace_bytes, st, engine == PCV_ENGINE_TCGEN05_F16);
  }

  SSPlan p;
  if (make_plan(t, M, &p) != PCV_OK) {
    set_error("score_select: dim %d unsupported", t->dim);
    return PCV_ERR_UNSUPPORTED;
  }
  if (workspace == nullptr || workspace_bytes < p.ws_bytes) {
    set_error("score_select: workspace too small (%zu < %zu)", workspace_bytes, p.ws_bytes);
    return PCV_ERR_WORKSPACE;
  }
  float *pv = reinterpret_cast<float *>(static_cast<char *>(workspace) + ss_ws_head(M));
  int32_t *pi = reinterpret_cast<int32_t *>(pv + (size_t)p.n_split * M);

  rc = opts->mode == PCV_SELECT_GREEDY ? dispatch_dim<SS_GREEDY>(t, p, Q, M, nullptr, pv, pi, nullptr, st)
                                       : dispatch_dim<SS_EXPRACE_NOISE>(t, p, Q, M, opts->noise, pv, pi, nullptr, st);
  if (rc != PCV_OK) return rc;
  int threads = 256;
  select_finalize_kernel<<<(unsigned)((M + threads - 1) / threads), threads, 0, st>>>(
      pv, pi, p.n_split, M, t->row_offset, out_idx, out_val);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

int pcv_score_logits(const pcv_table *th, const float *Q, int64_t M, float *out,
                     pcv_stream_t stream) {
  PCV_CHECK_ARG(th && Q && out, "NULL pointer");
  PCV_CHECK_ARG(M > 0, "M must be > 0");
  const Table *t = reinterpret_cast<const Table *>(th);
  PCV_CHECK_ARG(t->n_rows < 0x7fffffffLL, "shard larger than 2^31-1 rows");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  SSPlan p;
  if (make_plan(t, M, &p) != PCV_OK) {
    set_error("score_logits: dim %d unsupported", t->dim);
    return PCV_ERR_UNSUPPORTED;
  }
  return dispatch_dim<SS_LOGITS>(t, p, Q, M, nullptr, nullptr, nullptr, out, (cudaStream_t)stream);
}

int pcv_vp_pack_keys(const float *vals, const int64_t *idx, int64_t M, int64_t *keys, pcv_stream_t stream) {
  PCV_CHECK_ARG(vals && idx && keys, "NULL pointer");
  PCV_CHECK_ARG(M > 0, "M must be > 0");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  vp_pack_keys_kernel<<<(unsigned)((M + 255) / 256), 256, 0, (cudaStream_t)stream>>>(vals, idx, M,
                                                                                     reinterpret_cast<long long *>(keys));
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

int pcv_vp_unpack_keys(const int64_t *keys, int64_t M, int64_t *out_idx, float *out_val, pcv_stream_t stream) {
  PCV_CHECK_ARG(keys && out_idx, "NULL pointer");
  PCV_CHECK_ARG(M > 0, "M must be > 0");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  vp_unpack_keys_kernel<<<(unsigned)((M + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const long long *>(keys), M, out_idx, out_val);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

}  // extern "C"
