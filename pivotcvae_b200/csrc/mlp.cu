// mlp.cu — fused MLP blocks: gather/concat/one-hot prologue -> Linear+activation
// chain -> optional Gaussian reparameterisation epilogue, one kernel per block.
//
// Replaces (reference file:line)
//   cvae.py:85-92          get_condition (one-hot of the click count)      -> PCV_SEG_ONEHOT
//   pivotcvae.py:253,258   nn.Embedding gathers                            -> PCV_SEG_GATHER
//   pivotcvae.py:159-174   encode   [emb, c, u] -> enc_i (LeakyReLU) -> mu | logvar
//   pivotcvae.py:229-240   get_prior [c, u]     -> prior_i (LeakyReLU) -> mu | logvar
//   pivotcvae.py:204-210   PSM      [z, c, u]   -> psm_i (LeakyReLU except last)
//   pivotcvae.py:214-224   SCM      [z, c, pivot, u] -> scm_i; pivot row to slot 0 of rx
//   listcvae.py:106-119    decoder  [z, c, u]
//   cvae.py:79-83          reparametrize: z = eps * exp(0.5*logvar) + mu
//   env/response_model.py:76-87  response MLP (whole-vector L2 normalise, ReLU)
//
// Arithmetic contract: y[n] = (fma-chain over k ascending of x[k]*W[n][k], from 0) + b[n],
// i.e. the K loop is never split, so results are bit-identical to the CPU oracle.
//
// Layout: a CTA owns BM = 8/16/32 batch rows; activations ping-pong between two
// transposed shared-memory buffers actT[k][row]; each layer's weights stream through
// a double-buffered [32][256] shared-memory stage (transposed on the fly from
// nn.Linear's [n_out][n_in], prefetched one chunk ahead in registers); a thread
// accumulates an 8-row x CT-column register tile.
#include "mlp_common.cuh"
#include "tc_common.cuh"   // mbarrier / TMA bulk-copy helpers

namespace pcv {

// Prologue shared by both kernels: assemble x0 = [segments] into actA (transposed: element e of
// row r at actA[e * (BM + 4) + r]), segment-wide L2 normalisation, optional copies to HBM.
template <int THREADS, int BM, class Sync>
__device__ __forceinline__ void mlp_prologue(const MlpParams &P, int64_t B, float *actA, int64_t b0, int tid, Sync sync,
                                             bool write_hbm = true, int pad_to = 0) {
  constexpr int ALD = BM + 4;
  const pcv_mlp_desc &d = P.d;

    constexpr int TPR = THREADS / BM;  // threads per row
    const int row = tid / TPR, sub = tid % TPR;
    const int64_t b = b0 + row;
    float *x = actA + row;                 // element e at x[e * ALD]
    if (b < B) {
      for (int s = 0; s < d.n_segments; ++s) {
        const pcv_segment &sg = d.seg[s];
        float *xs = x + P.seg_off[s] * ALD;
        if (sg.kind == PCV_SEG_DENSE) {
          const float *src = (const float *)sg.ptr + b * sg.width;
          for (int e = sub; e < sg.width; e += TPR) xs[e * ALD] = src[e];
        } else if (sg.kind == PCV_SEG_ONEHOT) {
          const float *r = (const float *)sg.ptr + b * sg.count;
          float sum = 0.f;
          for (int l = 0; l < sg.count; ++l) sum += r[l];
          const int hot = (int)sum;  // .to(torch.long) truncates (cvae.py:91)
          for (int e = sub; e <= sg.count; e += TPR) xs[e * ALD] = (e == hot) ? 1.f : 0.f;
        } else {  // GATHER
          const float *tab = (const float *)sg.ptr;
          const int n = sg.count * sg.width;
          for (int e = sub; e < n; e += TPR) {
            const int c = e / sg.width, k = e - c * sg.width;
            xs[e * ALD] = tab[sg.idx[b * sg.count + c] * (int64_t)sg.width + k];
          }
        }
      }
    } else {
      for (int e = sub; e < P.n_in0; e += TPR) x[e * ALD] = 0.f;
    }
    for (int e = P.n_in0 + sub; e < pad_to; e += TPR) x[e * ALD] = 0.f;   // k padding of the first layer (cluster engine)
    sync();
    // segment-wide L2 normalisation (F.normalize eps=1e-12), sequential sum order
    for (int s = 0; s < d.n_segments; ++s) {
      if (d.seg[s].norm != PCV_NORM_SEGMENT) continue;
      const int w = P.seg_off[s + 1] - P.seg_off[s];
      float *xs = x + P.seg_off[s] * ALD;
      float ss = 0.f;
      for (int e = 0; e < w; ++e) ss = fmaf(xs[e * ALD], xs[e * ALD], ss);  // every thread of the row: same value
      const float nrm = fmaxf(sqrtf(ss), 1e-12f);
      sync();
      for (int e = sub; e < w; e += TPR) xs[e * ALD] = xs[e * ALD] / nrm;
      sync();
    }
    if (b < B && write_hbm) {
      if (d.x0) {
        float *dst = d.x0 + b * P.n_in0;
        for (int e = sub; e < P.n_in0; e += TPR) dst[e] = x[e * ALD];
      }
      if (d.copy_seg >= 0) {
        const int w = P.seg_off[d.copy_seg + 1] - P.seg_off[d.copy_seg];
        const float *xs = x + P.seg_off[d.copy_seg] * ALD;
        float *dst = d.out + b * d.out_ld;
        for (int e = sub; e < w; e += TPR) dst[e] = xs[e * ALD];
      }
    }
  }

// Reparameterisation epilogue (cvae.py:79-83): z = eps * exp(0.5 * logvar) + mu from the last layer's
// [mu | logvar] still in shared memory.
template <int THREADS, int BM>
__device__ __forceinline__ void mlp_reparam(const pcv_mlp_desc &d, const float *cur, int64_t b0, int64_t B, int tid) {
  constexpr int ALD = BM + 4;
  const int Z = d.latent;
  const uint64_t rng_off = d.offset + (d.offset_dev ? *d.offset_dev : 0ull);
  for (int e = tid; e < BM * Z; e += THREADS) {
    const int row = e / Z, j = e - row * Z;
    const int64_t b = b0 + row;
    if (b >= B) continue;
    const float mu = cur[j * ALD + row];
    const float lv = cur[(Z + j) * ALD + row];
    float eps;
    if (d.eps) {
      eps = d.eps[b * Z + j];
    } else {
      float n4[4];
      normal4(d.seed, rng_off, b, j >> 2, n4);
      eps = n4[j & 3];
    }
    const float sd = pcv_expf(lv * 0.5f);
    d.z[b * Z + j] = eps * sd + mu;
    if (d.eps_out) d.eps_out[b * Z + j] = eps;
  }
}

// Thread mapping: THREADS = (256/CT column groups) x (row groups of RT rows); a thread owns
// CT adjacent output columns x RT batch rows.  Small batches use <CT=1, RT=4, 512 threads>
// (8 rows per CTA, 16 warps per SM to hide the shared-memory latency); larger ones
// <CT=2|4, RT=8, 256 threads> (16 / 32 rows per CTA).
// Activations live TRANSPOSED in shared memory (actT[k][row]) so a thread's 8 rows
// are two broadcast LDS.128; the weight stage wst[kk][n] is read conflict-free.
// Weight chunks are prefetched into registers one chunk ahead (across column blocks
// and layers) and double-buffered in shared memory: one __syncthreads per chunk.
template <int CT, int RT, int THREADS>
__device__ __forceinline__ void mlp_block(const MlpParams &P, int64_t B, float *smem) {
  constexpr int CG = MLP_NB / CT;          // column groups (threads along n)
  constexpr int BM = RT * (THREADS / CG);  // batch rows per CTA
  constexpr int ALD = BM + 4;              // actT row stride (floats)
  constexpr int MLP_WLD = (CT == 1) ? MLP_NB + 1 : MLP_NB + 4;
  constexpr int NV4 = MLP_NB * MLP_KC / 4 / THREADS;   // float4 pieces of a weight chunk staged per thread
  constexpr int NV1 = MLP_NB * MLP_KC / THREADS;       // scalar pieces (ragged chunks)
  const int ld = P.ld;              // max width (multiple of 4)
  float *actA = smem;               // [ld][ALD]
  float *actB = actA + ld * ALD;
  float *wst = actB + ld * ALD;     // [2][MLP_KC][MLP_WLD]  (actB end is 16B-aligned: ld, ALD multiples of 4)

  const int tid = threadIdx.x;
  const int cg = tid % CG, rg = tid / CG;
  const int64_t b0 = (int64_t)blockIdx.x * BM;
  const pcv_mlp_desc &d = P.d;

  // ---------------- weight-chunk stream (layer, column block, k-chunk) ----------------
  int pl = 0, pnb = 0, pkc = 0;     // position of the chunk held in wv
  // Coalesced staging: MLP_KC/4 consecutive threads read one contiguous row segment W[n][kc..kc+MLP_KC-1]
  // (a per-thread-row pattern costs 32 L1 wavefronts per warp load: it was the bottleneck).
  float wv[NV1];
  bool wvec = true;   // layout of wv: float4 pieces (full, 16B-aligned chunk) or scalars (ragged chunk)
  auto fetch = [&](int l, int nb, int kc) {
    const int K = d.layer[l].n_in, NO = d.layer[l].n_out;
    wvec = (kc + MLP_KC <= K) && ((K & 3) == 0);
    if (wvec) {
#pragma unroll
      for (int i = 0; i < NV4; ++i) {
        const int f = tid + THREADS * i;
        const int n = nb + f / (MLP_KC / 4), c = f % (MLP_KC / 4);
        float4 t4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (n < NO) t4 = __ldg(reinterpret_cast<const float4 *>(d.layer[l].W + (int64_t)n * K + kc) + c);
        wv[4 * i] = t4.x; wv[4 * i + 1] = t4.y; wv[4 * i + 2] = t4.z; wv[4 * i + 3] = t4.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < NV1; ++i) {
        const int e = tid + THREADS * i;
        const int n = nb + e / MLP_KC, k = kc + e % MLP_KC;
        wv[i] = (n < NO && k < K) ? __ldg(d.layer[l].W + (int64_t)n * K + k) : 0.f;
      }
    }
  };
  auto stage = [&](float *ws) {   // registers -> transposed stage ws[kk][n]
    if (wvec) {
#pragma unroll
      for (int i = 0; i < NV4; ++i) {
        const int f = tid + THREADS * i;
        const int n = f / (MLP_KC / 4), k = (f % (MLP_KC / 4)) * 4;
#pragma unroll
        for (int j = 0; j < 4; ++j) ws[(k + j) * MLP_WLD + n] = wv[4 * i + j];
      }
    } else {
#pragma unroll
      for (int i = 0; i < NV1; ++i) {
        const int e = tid + THREADS * i;
        ws[(e % MLP_KC) * MLP_WLD + e / MLP_KC] = wv[i];
      }
    }
  };
  auto advance = [&]() {  // -> false when the stream is exhausted
    pkc += MLP_KC;
    if (pkc >= d.layer[pl].n_in) {
      pkc = 0;
      pnb += MLP_NB;
      if (pnb >= d.layer[pl].n_out) { pnb = 0; ++pl; }
    }
    return pl < d.n_layers;
  };
  fetch(0, 0, 0);  // in flight during the prologue
  // The whole weight set of the block (a few hundred KB) is requested into L2 up front, one
  // 128-byte line per prefetch, so the chunk-by-chunk loads below hit L2 instead of paying the
  // HBM latency once per chunk when the weights are cold (e.g. after an L2 flush).
  for (int l = 0; l < d.n_layers; ++l) {
    const char *wb = reinterpret_cast<const char *>(d.layer[l].W);
    const int64_t bytes = (int64_t)d.layer[l].n_in * d.layer[l].n_out * 4;
    for (int64_t o = (int64_t)tid * 128; o < bytes; o += (int64_t)THREADS * 128)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(wb + o));
  }

  mlp_prologue<THREADS, BM>(P, B, actA, b0, tid, [] { __syncthreads(); });

  // ---------------- layers ----------------
  float *cur = actA, *nxt = actB;
  int buf = 0;
  bool more = true;
  for (int l = 0; l < d.n_layers; ++l) {
    const pcv_linear L = d.layer[l];
    const bool last = (l == d.n_layers - 1);
    const int K = L.n_in;
    for (int nb = 0; nb < L.n_out; nb += MLP_NB) {
      float acc[RT][CT];
#pragma unroll
      for (int r = 0; r < RT; ++r)
#pragma unroll
        for (int c = 0; c < CT; ++c) acc[r][c] = 0.f;

      for (int kc = 0; kc < K; kc += MLP_KC) {
        float *ws = wst + buf * (MLP_KC * MLP_WLD);
        stage(ws);
        __syncthreads();
        if (more) {
          more = advance();
          if (more) fetch(pl, pnb, pkc);   // next chunk's loads fly during this chunk's FMAs
        }
        const int kmax = (nb + cg * CT < L.n_out) ? min(MLP_KC, K - kc) : 0;   // idle column groups skip the FMAs
        const float *ap = cur + (size_t)kc * ALD + rg * RT;
        // operands of step kk: RT activations (broadcast LDS.128) + CT weights
        auto load_ops = [&](int kk, float (&a)[RT], float (&w)[CT]) {
#pragma unroll
          for (int v = 0; v < RT / 4; ++v) {
            const float4 t4 = *reinterpret_cast<const float4 *>(ap + kk * ALD + 4 * v);
            a[4 * v] = t4.x; a[4 * v + 1] = t4.y; a[4 * v + 2] = t4.z; a[4 * v + 3] = t4.w;
          }
          if (CT == 4) {
            const float4 t4 = *reinterpret_cast<const float4 *>(ws + kk * MLP_WLD + cg * 4);
            w[0] = t4.x; w[1 % CT] = t4.y; w[2 % CT] = t4.z; w[3 % CT] = t4.w;
          } else if (CT == 2) {
            const float2 t2 = *reinterpret_cast<const float2 *>(ws + kk * MLP_WLD + cg * 2);
            w[0] = t2.x; w[1 % CT] = t2.y;
          } else {
            w[0] = ws[kk * MLP_WLD + cg];
          }
        };
        auto fma_ops = [&](const float (&a)[RT], const float (&w)[CT]) {
#pragma unroll
          for (int r = 0; r < RT; ++r)
#pragma unroll
            for (int c = 0; c < CT; ++c) acc[r][c] = fmaf(a[r], w[c], acc[r][c]);
        };
        if (kmax == MLP_KC) {
          // full chunk: explicit software pipeline, the operands of steps kk+1 and kk+2 are in flight
          // while step kk's FMAs issue (shared-memory latency ~30 cycles, only 2-4 warps per scheduler)
          float a0[RT], a1[RT], a2[RT], w0[CT], w1[CT], w2[CT];
          load_ops(0, a0, w0);
          load_ops(1, a1, w1);
#pragma unroll
          for (int kk = 0; kk < MLP_KC; kk += 3) {
            if (kk + 2 < MLP_KC) load_ops(kk + 2, a2, w2);
            fma_ops(a0, w0);
            if (kk + 3 < MLP_KC) load_ops(kk + 3, a0, w0);
            if (kk + 1 < MLP_KC) fma_ops(a1, w1);
            if (kk + 4 < MLP_KC) load_ops(kk + 4, a1, w1);
            if (kk + 2 < MLP_KC) fma_ops(a2, w2);
          }
        } else {
          for (int kk = 0; kk < kmax; ++kk) {
            float a[RT], w[CT];
            load_ops(kk, a, w);
            fma_ops(a, w);
          }
        }
        buf ^= 1;
      }
      // epilogue of this column block: bias + activation -> nxt (+ HBM)
#pragma unroll
      for (int c = 0; c < CT; ++c) {
        const int n = nb + cg * CT + c;
        if (n < L.n_out) {
          const float bias = __ldg(L.b + n);
          float v[RT];
#pragma unroll
          for (int r = 0; r < RT; ++r) v[r] = apply_act(acc[r][c] + bias, L.act);
          float *np = nxt + (size_t)n * ALD + rg * RT;
#pragma unroll
          for (int q4 = 0; q4 < RT / 4; ++q4)
            *reinterpret_cast<float4 *>(np + 4 * q4) = make_float4(v[4 * q4], v[4 * q4 + 1], v[4 * q4 + 2], v[4 * q4 + 3]);
#pragma unroll
          for (int r = 0; r < RT; ++r) {
            const int64_t b = b0 + rg * RT + r;
            if (b < B) {
              if (last) d.out[b * d.out_ld + d.out_col0 + n] = v[r];
              else if (d.acts[l]) d.acts[l][b * L.n_out + n] = v[r];
            }
          }
        }
      }
    }
    float *t = cur; cur = nxt; nxt = t;
  }
  __syncthreads();

  if (d.latent > 0) mlp_reparam<THREADS, BM>(d, cur, b0, B, tid);
}

template <int CT, int RT, int THREADS>
__global__ void __launch_bounds__(THREADS)
mlp_fwd_kernel(const MlpParams P, int64_t B) {
  extern __shared__ __align__(16) float smem[];
  mlp_block<CT, RT, THREADS>(P, B, smem);
}

// Two chained blocks in one launch (e.g. prior -> reparameterise -> PSM, pivotcvae.py:279-291 +
// 204-210): block B's prologue reads what block A just wrote for the SAME batch rows (z), so a
// CTA-level fence + barrier is all the ordering it needs.
template <int CT, int RT, int THREADS>
__global__ void __launch_bounds__(THREADS)
mlp_fwd2_kernel(const MlpParams2 P, int64_t B) {
  extern __shared__ __align__(16) float smem[];
  mlp_block<CT, RT, THREADS>(P.a, B, smem);
  __threadfence_block();
  __syncthreads();
  mlp_block<CT, RT, THREADS>(P.b, B, smem);
}

// ===========================================================================
// Packed-weight cluster engine (inference).  The streaming engine above makes every CTA pull the
// whole weight set of the block through L2 (128 CTAs x 360 KB at B=1024): measured L2-bound.
// Here a CLUSTER of 4 CTAs owns 32 batch rows and splits every layer's output columns in 64-wide
// blocks (block j -> CTA j mod 4), so each CTA streams a quarter of the weights:
//   * weights are pre-tiled once by pcv_mlp_pack into the shared-memory image a k-chunk needs:
//     tile (block j, chunk kc) = [32][nbw] floats, element (kk, n) = W[64 j + n][kc + kk] (zero
//     padded), nbw = min(64, round_up32(n_out - 64 j)) -> a chunk is ONE TMA bulk copy issued by a
//     producer warp into an 8-stage mbarrier ring (no per-chunk __syncthreads, no weight LDG/STS);
//   * 8 compute warps, warp = 4 rows, lane = 2 columns (a single warp per scheduler issues an FFMA
//     only every other cycle: measured, so two warps share each scheduler);
//   * a block's outputs are written straight into the next layer's activation buffer of ALL four
//     CTAs (st.shared::cluster) and one cluster barrier per layer publishes them;
//   * narrow layers (<= 64 outputs: heads, last layers) split the ROWS over the cluster instead
//     (rank r = rows 8r..8r+7, warp = row, lane = column), every rank streaming the small tiles.
// Same arithmetic contract (sequential-k FMA chain) -> bit-identical to the streaming engine.
// ===========================================================================
#ifdef PCV_TC_TRACE
__device__ long long g_mlp_trace[4][32];   // [cluster rank of cluster 0][event]
#define MLP_TRACE(i) do { if (blockIdx.x < 4 && threadIdx.x == 0) g_mlp_trace[blockIdx.x][i] = clock64(); } while (0)
#else
#define MLP_TRACE(i) do { } while (0)
#endif

constexpr int MLPC_CL = 4;                 // CTAs per cluster
constexpr int MLPC_BN = 64;                // output columns per block
constexpr int MLPC_BM = 32;                // batch rows per cluster
constexpr int MLPC_ALD = MLPC_BM + 4;      // activation row stride (floats)
constexpr int MLPC_STAGES = 8;
constexpr int MLPC_TILE_FLOATS = MLP_KC * MLPC_BN;   // 8 KB
constexpr int MLPC_ROWSPLIT_MAX = 64;      // layers up to this wide split the rows, not the columns, over the cluster
constexpr int MLPC_NC = 256;               // compute threads: 8 warps = 8 row groups of 4 rows

__host__ __device__ __forceinline__ int mlpc_nbw(int n_out, int nb) {
  const int w = ((n_out - nb) + 31) & ~31;
  return w < MLPC_BN ? w : MLPC_BN;
}
__host__ __device__ __forceinline__ int64_t mlpc_packed_floats(int n_in, int n_out) {
  const int64_t kpad = (n_in + MLP_KC - 1) / MLP_KC * MLP_KC;
  int64_t cols = 0;
  for (int nb = 0; nb < n_out; nb += MLPC_BN) cols += mlpc_nbw(n_out, nb);
  return kpad * cols;
}

__global__ void mlp_pack_kernel(const float *__restrict__ W, int K, int NO, float *__restrict__ Wp, int64_t total) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const int64_t kpad = (K + MLP_KC - 1) / MLP_KC * MLP_KC;
  const int j = (int)(e / (kpad * MLPC_BN));           // every block before the last is 64 wide
  const int nb = j * MLPC_BN;
  const int nbw = mlpc_nbw(NO, nb);
  const int64_t local = e - (int64_t)j * kpad * MLPC_BN;
  const int k = (int)(local / nbw), n = (int)(local % nbw);   // tile kc = k / 32 at kc * 32 * nbw, row kk = k % 32
  Wp[e] = (nb + n < NO && k < K) ? W[(int64_t)(nb + n) * K + k] : 0.f;
}

__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void st_cluster_f4(uint32_t local_addr, uint32_t rank, float4 v) {
  uint32_t ra;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(local_addr), "r"(rank));
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(ra), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}

__device__ __forceinline__ void st_cluster_f1(uint32_t local_addr, uint32_t rank, float v) {
  uint32_t ra;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(local_addr), "r"(rank));
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(ra), "f"(v) : "memory");
}

template <int ST>
__device__ __forceinline__ void mlpc_block(const MlpParams &P, int64_t B, float *actA, float *actB, const float *stage,
                                           unsigned long long *full, unsigned long long *empty, uint32_t &g,
                                           uint32_t crank) {
  constexpr int CT = 2, RT = 4;
  const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;   // warp = row group (4 rows), lane = 2 columns
  const int64_t b0 = (int64_t)(blockIdx.x / MLPC_CL) * MLPC_BM;
  const pcv_mlp_desc &d = P.d;
  auto csync = [] { asm volatile("bar.sync 1, %0;" ::"n"(MLPC_NC) : "memory"); };

  // every CTA of the cluster assembles the (same) input rows in its own buffer; rank 0 writes the HBM copies
  MLP_TRACE(1);
  // every k range is padded to a multiple of 32 with zeros (activation rows here and in the epilogues
  // below, weight tiles by pcv_mlp_pack): adding a*0 to a sequential FMA chain never changes it
  mlp_prologue<MLPC_NC, MLPC_BM>(P, B, actA, b0, tid, csync, crank == 0, (P.n_in0 + MLP_KC - 1) / MLP_KC * MLP_KC);
  MLP_TRACE(2);

  float *cur = actA, *nxt = actB;
  for (int l = 0; l < d.n_layers; ++l) {
    const pcv_linear L = d.layer[l];
    const bool last = (l == d.n_layers - 1);
    const int K = L.n_in;
    if (L.n_out > MLPC_ROWSPLIT_MAX) {
      // ---- wide layer: column split, 64-wide block j -> rank j mod 4; warp = 4 rows, lane = 2 columns
      for (int nb = (int)crank * MLPC_BN; nb < L.n_out; nb += MLPC_CL * MLPC_BN) {
        const int nbw = mlpc_nbw(L.n_out, nb);
        const bool active = lane * CT < nbw;   // lanes past the (padded) block only keep the ring moving
        // accumulators as fp32x2 pairs of adjacent rows: acc2[p][c] = (row 2p, row 2p+1) of column c
        unsigned long long acc2[RT / 2][CT];
#pragma unroll
        for (int r = 0; r < RT / 2; ++r)
#pragma unroll
          for (int c = 0; c < CT; ++c) acc2[r][c] = 0ull;
        for (int kc = 0; kc < K; kc += MLP_KC, ++g) {
          const int s = g % ST;
          mbar_wait(&full[s], (g / ST) & 1);
          if (active) {
            const float *ws = stage + (size_t)s * MLPC_TILE_FLOATS + lane * CT;
            const float *ap = cur + (size_t)kc * MLPC_ALD + wrp * RT;
            auto load_ops = [&](int kk, float (&a)[RT], float (&w)[CT]) {
              const float4 a0 = *reinterpret_cast<const float4 *>(ap + kk * MLPC_ALD);
              a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w;
              const float2 w2 = *reinterpret_cast<const float2 *>(ws + kk * nbw);
              w[0] = w2.x; w[1] = w2.y;
            };
            // 4 FFMA2 per k-step: (rows 0,1 | rows 2,3) x (column 0 | column 1), the weight broadcast to both halves
            auto fma_ops = [&](const float (&a)[RT], const float (&w)[CT]) {
              const unsigned long long a01 = pack2(a[0], a[1]), a23 = pack2(a[2], a[3]);
              const unsigned long long w0 = pack2(w[0], w[0]), w1 = pack2(w[1], w[1]);
              ffma2(acc2[0][0], a01, w0);
              ffma2(acc2[0][1], a01, w1);
              ffma2(acc2[1][0], a23, w0);
              ffma2(acc2[1][1], a23, w1);
            };
            // two warps per scheduler: the operands of the next three k-steps are in flight while
            // this step's FMAs issue
            float a0[RT], a1[RT], a2[RT], a3[RT], w0[CT], w1[CT], w2[CT], w3[CT];
            load_ops(0, a0, w0);
            load_ops(1, a1, w1);
            load_ops(2, a2, w2);
#pragma unroll
            for (int kk = 0; kk < MLP_KC; kk += 4) {
              load_ops(kk + 3, a3, w3);
              fma_ops(a0, w0);
              if (kk + 4 < MLP_KC) load_ops(kk + 4, a0, w0);
              fma_ops(a1, w1);
              if (kk + 5 < MLP_KC) load_ops(kk + 5, a1, w1);
              fma_ops(a2, w2);
              if (kk + 6 < MLP_KC) load_ops(kk + 6, a2, w2);
              fma_ops(a3, w3);
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty[s]);   // this warp is done reading the stage
        }
        float acc[RT][CT];
#pragma unroll
        for (int r = 0; r < RT / 2; ++r)
#pragma unroll
          for (int c = 0; c < CT; ++c) unpack2(acc2[r][c], acc[2 * r][c], acc[2 * r + 1][c]);
        // bias + activation -> the next layer's buffer of all four CTAs (+ HBM); padded columns -> 0
#pragma unroll
        for (int c = 0; c < CT; ++c) {
          const int n = nb + lane * CT + c;
          if (n < nb + nbw) {
            const bool real = n < L.n_out;
            const float bias = real ? __ldg(L.b + n) : 0.f;
            float v[RT];
#pragma unroll
            for (int r = 0; r < RT; ++r) v[r] = real ? apply_act(acc[r][c] + bias, L.act) : 0.f;
            const uint32_t np = smem_u32(nxt + (size_t)n * MLPC_ALD + wrp * RT);
#pragma unroll
            for (uint32_t t = 0; t < MLPC_CL; ++t) st_cluster_f4(np, t, make_float4(v[0], v[1], v[2], v[3]));
            if (real) {
#pragma unroll
              for (int r = 0; r < RT; ++r) {
                const int64_t b = b0 + wrp * RT + r;
                if (b < B) {
                  if (last) d.out[b * d.out_ld + d.out_col0 + n] = v[r];
                  else if (d.acts[l]) d.acts[l][b * L.n_out + n] = v[r];
                }
              }
            }
          }
        }
      }
    } else {
      // ---- narrow layer: a column split would idle three CTAs (and most lanes), so the ROWS are split:
      // rank r computes rows 8r..8r+7 for every column; warp = one row, lane = columns lane (+32)
      const int row = (int)crank * (MLPC_BM / MLPC_CL) + wrp;
      for (int nb = 0; nb < L.n_out; nb += MLPC_BN) {
        const int nbw = mlpc_nbw(L.n_out, nb);
        const bool two = nbw > 32;
        float acc0 = 0.f, acc1 = 0.f;
        for (int kc = 0; kc < K; kc += MLP_KC, ++g) {
          const int s = g % ST;
          mbar_wait(&full[s], (g / ST) & 1);
          const float *ws = stage + (size_t)s * MLPC_TILE_FLOATS + lane;
          const float *ap = cur + (size_t)kc * MLPC_ALD + row;
          if (two) {
#pragma unroll
            for (int kk = 0; kk < MLP_KC; ++kk) {
              const float a = ap[kk * MLPC_ALD];
              acc0 = fmaf(a, ws[kk * 64], acc0);
              acc1 = fmaf(a, ws[kk * 64 + 32], acc1);
            }
          } else {
#pragma unroll
            for (int kk = 0; kk < MLP_KC; ++kk) acc0 = fmaf(ap[kk * MLPC_ALD], ws[kk * 32], acc0);
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty[s]);
        }
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const int n = nb + lane + 32 * c;
          if (n < nb + nbw) {
            const bool real = n < L.n_out;
            const float v = real ? apply_act((c ? acc1 : acc0) + __ldg(L.b + n), L.act) : 0.f;
            const uint32_t np = smem_u32(nxt + (size_t)n * MLPC_ALD + row);
#pragma unroll
            for (uint32_t t = 0; t < MLPC_CL; ++t) st_cluster_f1(np, t, v);
            const int64_t b = b0 + row;
            if (real && b < B) {
              if (last) d.out[b * d.out_ld + d.out_col0 + n] = v;
              else if (d.acts[l]) d.acts[l][b * L.n_out + n] = v;
            }
          }
        }
      }
    }
    MLP_TRACE(3 + 2 * l);
    cluster_sync_all();   // every CTA's part of nxt has landed everywhere; cur is no longer read anywhere
    MLP_TRACE(4 + 2 * l);
    float *t = cur; cur = nxt; nxt = t;
  }
  if (d.latent > 0 && crank == 0) mlp_reparam<MLPC_NC, MLPC_BM>(d, cur, b0, B, tid);
}

// warps 0-7 compute; warp 8 streams this CTA's weight tiles of the whole launch (both blocks of a
// chain back to back: the second block's weights prefetch while the first one finishes)
// ST = stages of the weight ring: 8 (64 KB, deepest prefetch) when the launch is a single wave, 4 (32 KB) when there
// are more CTAs than SMs, so that TWO CTAs fit an SM (2 x ~107 KB) and one hides the other's barrier / TMA latencies
template <int ST>
__global__ void __cluster_dims__(MLPC_CL, 1, 1) __launch_bounds__(MLPC_NC + 32)
mlp_cluster_kernel(const MlpParams2 P, int n_blocks, int64_t B) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float *stage = reinterpret_cast<float *>(smem_raw);                               // [8][32][64]
  unsigned long long *full = reinterpret_cast<unsigned long long *>(stage + ST * MLPC_TILE_FLOATS);
  unsigned long long *empty = full + ST;
  float *actA = reinterpret_cast<float *>(empty + ST);                      // 16-byte aligned
  float *actB = actA + (size_t)P.a.ld * MLPC_ALD;
  const uint32_t crank = cluster_rank();
  MLP_TRACE(0);
  if (threadIdx.x == 0) {
    for (int s = 0; s < ST; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], MLPC_NC / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  cluster_sync_all();   // nobody writes into a peer's shared memory before that peer is running
  if (threadIdx.x >= MLPC_NC) {
    // The cluster barriers count every thread of the cluster, so this warp takes part in each of
    // them, in the compute threads' order (one per layer, one between chained blocks).  It must
    // never BLOCK on a barrier before the tiles the compute threads need to reach it are issued:
    // arrive(e) follows the issue of layer e's tiles, and the matching wait is deferred until
    // the next layer's tiles are issued too (so the producer runs up to one layer ahead).
    // cold start (weights not in L2, e.g. the first call after other work evicted them): request this
    // rank's tiles of the whole launch into L2 up front, clusters taking turns over the tile list
    {
      const int lane = threadIdx.x & 31;
      const unsigned ncl = gridDim.x / MLPC_CL, cl = blockIdx.x / MLPC_CL;
      unsigned t = 0;
      for (int blk = 0; blk < n_blocks; ++blk) {
        const pcv_mlp_desc &d = blk ? P.b.d : P.a.d;
        for (int l = 0; l < d.n_layers; ++l) {
          const int K = d.layer[l].n_in, NO = d.layer[l].n_out;
          const int64_t kpad = (K + MLP_KC - 1) / MLP_KC * MLP_KC;
          const bool rowsplit = NO <= MLPC_ROWSPLIT_MAX;
          for (int nb = rowsplit ? 0 : (int)crank * MLPC_BN; nb < NO; nb += (rowsplit ? 1 : MLPC_CL) * MLPC_BN, ++t) {
            if (t % 8 != cl % 8 && ncl >= 8) continue;
            const char *src = reinterpret_cast<const char *>(d.layer[l].Wp + (int64_t)nb * kpad);
            const int64_t bytes = kpad * mlpc_nbw(NO, nb) * (int64_t)sizeof(float);
            for (int64_t o = (int64_t)lane * 128; o < bytes; o += 32 * 128)
              asm volatile("prefetch.global.L2 [%0];" ::"l"(src + o));
          }
        }
      }
    }
    uint32_t g = 0;
    bool pending = false;
    auto event = [&]() {
      __syncwarp();
      if (pending) asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
      asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
      pending = true;
    };
    for (int blk = 0; blk < n_blocks; ++blk) {
      const pcv_mlp_desc &d = blk ? P.b.d : P.a.d;
      if (blk) event();   // the barrier between chained blocks
      for (int l = 0; l < d.n_layers; ++l) {
        if (threadIdx.x == MLPC_NC) {
          const int K = d.layer[l].n_in, NO = d.layer[l].n_out;
          const int64_t kpad = (K + MLP_KC - 1) / MLP_KC * MLP_KC;
          const bool rowsplit = NO <= MLPC_ROWSPLIT_MAX;   // every rank needs every block of a narrow layer
          for (int nb = rowsplit ? 0 : (int)crank * MLPC_BN; nb < NO; nb += (rowsplit ? 1 : MLPC_CL) * MLPC_BN) {
            const int nbw = mlpc_nbw(NO, nb);
            const float *src = d.layer[l].Wp + (int64_t)nb * kpad;
            const uint32_t bytes = (uint32_t)(MLP_KC * nbw * sizeof(float));
            for (int kc = 0; kc < K; kc += MLP_KC, ++g) {
              const int s = g % ST;
              mbar_wait(&empty[s], ((g / ST) & 1) ^ 1);
              mbar_expect_tx(&full[s], bytes);
              tma_bulk_load(stage + (size_t)s * MLPC_TILE_FLOATS, src + (int64_t)kc * nbw, bytes, &full[s]);
            }
          }
        }
        event();   // the barrier that ends layer l
      }
    }
    if (pending) asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
    return;
  }
  uint32_t g = 0;
  mlpc_block<ST>(P.a, B, actA, actB, stage, full, empty, g, crank);
  MLP_TRACE(20);
  if (n_blocks > 1) {
    // block B's prologue reads what rank 0 just wrote to HBM for the cluster's batch rows (z)
    __threadfence();
    cluster_sync_all();
    mlpc_block<ST>(P.b, B, actA, actB, stage, full, empty, g, crank);
  }
}

// KL(q||p) summed (train_generative.py:61) with analytic gradients; one CTA,
// fixed reduction order (deterministic).
__global__ void __launch_bounds__(1024)
kl_kernel(const float *__restrict__ mu, const float *__restrict__ lv, const float *__restrict__ pmu,
          const float *__restrict__ plv, int64_t n, float *__restrict__ kl_out,
          float *__restrict__ dmu, float *__restrict__ dlv, float *__restrict__ dpmu,
          float *__restrict__ dplv) {
  __shared__ float red[32];
  float acc = 0.f;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const float m = mu[i], v = lv[i], pm = pmu[i], pv = plv[i];
    const float ev = expf(v), ipv = expf(-pv), dm = m - pm;
    const float ratio = (ev + dm * dm) * ipv;
    acc += 1.f + v - pv - ratio;
    if (dmu) dmu[i] = dm * ipv;
    if (dlv) dlv[i] = -0.5f * (1.f - ev * ipv);
    if (dpmu) dpmu[i] = -dm * ipv;
    if (dplv) dplv[i] = -0.5f * (ratio - 1.f);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) *kl_out = -0.5f * v;
  }
}

}  // namespace pcv

using namespace pcv;

extern "C" {

static int mlp_prepare(const pcv_mlp_desc *d, MlpParams *Pp) {
  MlpParams &P = *Pp;
  PCV_CHECK_ARG(d != nullptr, "desc is NULL");
  PCV_CHECK_ARG(d->n_segments >= 1 && d->n_segments <= PCV_MAX_SEGMENTS, "bad n_segments");
  PCV_CHECK_ARG(d->n_layers >= 1 && d->n_layers <= PCV_MAX_LAYERS, "bad n_layers");
  PCV_CHECK_ARG(d->out != nullptr, "out is NULL");
  P.d = *d;
  int off = 0;
  for (int s = 0; s < d->n_segments; ++s) {
    const pcv_segment &sg = d->seg[s];
    PCV_CHECK_ARG(sg.ptr != nullptr, "segment pointer is NULL");
    P.seg_off[s] = off;
    if (sg.kind == PCV_SEG_DENSE) {
      PCV_CHECK_ARG(sg.width > 0, "dense segment width");
      off += sg.width;
    } else if (sg.kind == PCV_SEG_ONEHOT) {
      PCV_CHECK_ARG(sg.count > 0, "one-hot segment count");
      off += sg.count + 1;
    } else if (sg.kind == PCV_SEG_GATHER) {
      PCV_CHECK_ARG(sg.idx != nullptr && sg.width > 0 && sg.count > 0, "gather segment");
      off += sg.width * sg.count;
    } else {
      PCV_CHECK_ARG(false, "unknown segment kind");
    }
  }
  P.seg_off[d->n_segments] = off;
  P.n_in0 = off;
  int maxw = off;
  int prev = off;
  for (int l = 0; l < d->n_layers; ++l) {
    const pcv_linear &L = d->layer[l];
    PCV_CHECK_ARG(L.W && L.b, "layer weights are NULL");
    if (L.n_in != prev) {
      set_error("pcv_mlp_fwd: layer %d expects n_in=%d but receives %d", l, L.n_in, prev);
      return PCV_ERR_ARG;
    }
    PCV_CHECK_ARG(L.n_out > 0, "layer n_out");
    PCV_CHECK_ARG(((uintptr_t)L.W & 15) == 0, "layer weight must be 16-byte aligned");
    if (L.n_out > maxw) maxw = L.n_out;
    prev = L.n_out;
  }
  PCV_CHECK_ARG(maxw <= PCV_MAX_WIDTH, "layer wider than PCV_MAX_WIDTH");
  PCV_CHECK_ARG(d->copy_seg < d->n_segments, "copy_seg out of range");
  PCV_CHECK_ARG(d->out_ld >= d->out_col0 + prev, "out_ld too small");
  if (d->latent > 0) {
    PCV_CHECK_ARG(prev == 2 * d->latent, "reparam needs the last layer to emit 2*latent");
    PCV_CHECK_ARG(d->z != nullptr, "z is NULL");
  }
  P.ld = (maxw + 3) & ~3;
  return PCV_OK;
}

static bool mlp_saves(const MlpParams &P) {
  for (int l = 0; l < P.d.n_layers - 1; ++l)
    if (P.d.acts[l] != nullptr) return true;
  return P.d.x0 != nullptr;
}

// packed-weight cluster engine: 32 rows per cluster of 4 CTAs; k ranges / column blocks are zero-padded to multiples
// of 32; a grid of more than one wave gets the shallower weight ring
static size_t mlpc_smem(int64_t B, int ld, int sm_count, int *stages) {
  *stages = ((B + MLPC_BM - 1) / MLPC_BM * MLPC_CL > sm_count) ? 4 : MLPC_STAGES;
  return (size_t)*stages * MLPC_TILE_FLOATS * sizeof(float) + 2 * *stages * 8 + (size_t)2 * ld * MLPC_ALD * sizeof(float);
}
static int mlpc_ld(int ld) { return (ld + MLP_KC - 1) / MLP_KC * MLP_KC; }

// Validates the descriptors (b NULL = one block, then P->b = P->a; both blocks share the wider activation stride) and
// chooses the kernel: the one decision behind pcv_mlp_plan, pcv_mlp_fwd and pcv_mlp_fwd2.  It reads shapes and saved
// outputs, never a weight image.
static int mlp_plan(const pcv_mlp_desc *a, const pcv_mlp_desc *b, int64_t B, int engine, MlpParams2 *P, int *sm_count,
                    int *kernel) {
  PCV_CHECK_ARG(B > 0, "B must be > 0");
  PCV_CHECK_ARG(engine == PCV_MLP_EXACT || engine == PCV_MLP_TC || engine == PCV_MLP_AUTO, "unknown engine");
  int rc = mlp_prepare(a, &P->a);
  if (rc != PCV_OK) return rc;
  P->b = P->a;
  if (b && (rc = mlp_prepare(b, &P->b)) != PCV_OK) return rc;
  P->a.ld = P->b.ld = P->a.ld > P->b.ld ? P->a.ld : P->b.ld;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(sm_count, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
    cudaGetLastError();
    *sm_count = 148;   // no device (pcv_mlp_plan on a host without a GPU): a B200's count
  }
  int stages;
  if (mlp_saves(P->a) || mlp_saves(P->b))
    *kernel = PCV_MLP_KERNEL_STREAM;   // only the streaming engine writes x0 / acts
  else if (mlp_tc_takes(*P, B, engine))
    *kernel = PCV_MLP_KERNEL_TC;
  else
    *kernel = mlpc_smem(B, mlpc_ld(P->a.ld), *sm_count, &stages) <= 227 * 1024 ? PCV_MLP_KERNEL_CLUSTER
                                                                              : PCV_MLP_KERNEL_STREAM;
  return PCV_OK;
}

static int mlp_launch_cluster(MlpParams2 P2, int nblk, int64_t B, int sm_count, cudaStream_t st) {
  P2.a.ld = P2.b.ld = mlpc_ld(P2.a.ld);
  int stages;
  const size_t smem = mlpc_smem(B, P2.a.ld, sm_count, &stages);
  const unsigned grid = (unsigned)((B + MLPC_BM - 1) / MLPC_BM * MLPC_CL);
  if (stages == 4) {
    PCV_CUDA(cudaFuncSetAttribute(mlp_cluster_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    mlp_cluster_kernel<4><<<grid, MLPC_NC + 32, smem, st>>>(P2, nblk, B);
  } else {
    PCV_CUDA(cudaFuncSetAttribute(mlp_cluster_kernel<MLPC_STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    mlp_cluster_kernel<MLPC_STAGES><<<grid, MLPC_NC + 32, smem, st>>>(P2, nblk, B);
  }
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

static int mlp_launch_stream(const MlpParams2 &P2, int nblk, int64_t B, int sm_count, cudaStream_t st) {
  const int ld = P2.a.ld;
  // rows per CTA: 8 / 16 / 32 — small batches spread over more SMs (and use 16 warps per CTA)
  int CT = (B <= (int64_t)sm_count * 16) ? 1 : (B <= (int64_t)sm_count * 64 ? 2 : 4);
  auto smem_of = [&](int ct) { return (size_t)(2 * ld * (8 * ct + 4) + 2 * MLP_KC * MLP_WLD_MAX) * sizeof(float); };
  while (CT > 1 && smem_of(CT) > 227 * 1024) CT >>= 1;   // wide layers (up to PCV_MAX_WIDTH = 1024): fewer rows per CTA
  const int BM = 8 * CT;
  size_t smem = smem_of(CT);
  if (smem > 227 * 1024) {
    set_error("pcv_mlp_fwd: activations of width %d do not fit shared memory", ld);
    return PCV_ERR_UNSUPPORTED;
  }
  int64_t blocks = (B + BM - 1) / BM;
#define PCV_MLP_LAUNCH(CTv, RTv, THv)                                                                              \
  if (nblk == 2) {                                                                                                 \
    PCV_CUDA(cudaFuncSetAttribute(mlp_fwd2_kernel<CTv, RTv, THv>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    mlp_fwd2_kernel<CTv, RTv, THv><<<(unsigned)blocks, THv, smem, st>>>(P2, B);                                  \
  } else {                                                                                                         \
    PCV_CUDA(cudaFuncSetAttribute(mlp_fwd_kernel<CTv, RTv, THv>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    mlp_fwd_kernel<CTv, RTv, THv><<<(unsigned)blocks, THv, smem, st>>>(P2.a, B);                                 \
  }
  if (CT == 1) { PCV_MLP_LAUNCH(1, 4, 512) } else if (CT == 2) { PCV_MLP_LAUNCH(2, 8, 256) } else { PCV_MLP_LAUNCH(4, 8, 256) }
#undef PCV_MLP_LAUNCH
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

static int mlp_run(const pcv_mlp_desc *a, const pcv_mlp_desc *b, int64_t B, int engine, cudaStream_t st) {
  MlpParams2 P;
  int sm_count, kernel;
  int rc = mlp_plan(a, b, B, engine, &P, &sm_count, &kernel);
  if (rc != PCV_OK) return rc;
  const int nblk = b ? 2 : 1;
  // the planned kernel reads its weight image on every layer: a missing one is an error, not a fallback
  for (int blk = 0; blk < nblk && kernel != PCV_MLP_KERNEL_STREAM; ++blk)
    for (int l = 0; l < (blk ? P.b : P.a).d.n_layers; ++l) {
      const pcv_linear &L = (blk ? P.b : P.a).d.layer[l];
      if ((kernel == PCV_MLP_KERNEL_TC ? L.Wt : L.Wp) == nullptr) {
        set_error("pcv_mlp_fwd: block %d layer %d has no pcv_linear.%s, which the planned %s kernel reads", blk, l,
                  kernel == PCV_MLP_KERNEL_TC ? "Wt" : "Wp", kernel == PCV_MLP_KERNEL_TC ? "tc" : "cluster");
        return PCV_ERR_ARG;
      }
    }
  rc = check_arch();
  if (rc != PCV_OK) return rc;
  if (kernel == PCV_MLP_KERNEL_TC) return mlp_tc_launch(P, nblk, B, st);
  if (kernel == PCV_MLP_KERNEL_CLUSTER) return mlp_launch_cluster(P, nblk, B, sm_count, st);
  return mlp_launch_stream(P, nblk, B, sm_count, st);
}

int pcv_mlp_plan(const pcv_mlp_desc *a, const pcv_mlp_desc *b, int64_t B, int engine, int *kernel) {
  PCV_CHECK_ARG(kernel != nullptr, "kernel is NULL");
  MlpParams2 P;
  int sm_count;
  return mlp_plan(a, b, B, engine, &P, &sm_count, kernel);
}

int pcv_mlp_fwd(const pcv_mlp_desc *d, int64_t B, int engine, pcv_stream_t stream) {
  return mlp_run(d, nullptr, B, engine, (cudaStream_t)stream);
}

int pcv_mlp_fwd2(const pcv_mlp_desc *a, const pcv_mlp_desc *b, int64_t B, int engine, pcv_stream_t stream) {
  PCV_CHECK_ARG(b != nullptr, "desc b is NULL");
  return mlp_run(a, b, B, engine, (cudaStream_t)stream);
}

size_t pcv_mlp_packed_bytes(int n_in, int n_out) {
  if (n_in <= 0 || n_out <= 0) return 0;
  return (size_t)mlpc_packed_floats(n_in, n_out) * sizeof(float);
}

int pcv_mlp_pack(const float *W, int n_in, int n_out, float *packed, pcv_stream_t stream) {
  PCV_CHECK_ARG(W && packed, "NULL pointer");
  PCV_CHECK_ARG(n_in > 0 && n_out > 0 && n_in <= PCV_MAX_WIDTH && n_out <= PCV_MAX_WIDTH, "bad layer shape");
  PCV_CHECK_ARG(((uintptr_t)packed & 127) == 0, "packed buffer must be 128-byte aligned");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  const int64_t total = mlpc_packed_floats(n_in, n_out);
  mlp_pack_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(W, n_in, n_out, packed, total);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

#ifdef PCV_TC_TRACE
int pcv_debug_mlp_trace(long long *host4x32) {
  return (int)cudaMemcpyFromSymbol(host4x32, g_mlp_trace, sizeof(long long) * 4 * 32);
}
#endif

int pcv_kl_fwd_bwd(const float *mu, const float *logvar, const float *pmu, const float *plogvar,
                   int64_t n, float *kl_out, float *dmu, float *dlogvar, float *dpmu,
                   float *dplogvar, pcv_stream_t stream) {
  PCV_CHECK_ARG(mu && logvar && pmu && plogvar && kl_out, "NULL pointer");
  PCV_CHECK_ARG(n > 0, "n must be > 0");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  kl_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(mu, logvar, pmu, plogvar, n, kl_out, dmu, dlogvar,
                                                  dpmu, dplogvar);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

}  // extern "C"
