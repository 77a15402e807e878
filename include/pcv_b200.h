/*
 * pcv_b200.h — C ABI of libpcv_b200.so, the sm_100a slate-generation hot path.
 *
 * The reference (CharlieMat/PivotCVAE) has no FFI: its boundary is the Python
 * class API (models/cvae.py, models/pivotcvae.py, models/listcvae.py,
 * env/response_model.py, train_generative.py).  This header is the layer a
 * maintainer would bind *underneath* those classes (ctypes stub in
 * INTEGRATION.md).  Each entry point cites the reference lines it replaces.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller (torch), except
 *    descriptor structs (host) and out-params named *_host;
 *  - every op takes a cudaStream_t (as void*) and is asynchronous on it;
 *  - return 0 on success, <0 on error (pcv_last_error() gives the text);
 *  - no allocation inside ops: scratch comes from the caller through the
 *    *_workspace_bytes() queries.  The one exception is pcv_table_create, a
 *    one-off constructor: it synchronises the device and allocates the handle's
 *    packed table copies (freed by pcv_table_destroy); a failure there is an
 *    error, never a silent downgrade to a slower engine.  pcv_table_refresh
 *    brings those copies up to date on a stream without either;
 *  - float = IEEE binary32, indices = int64 (torch.long), row-major tensors.
 *  - there is no CPU fallback: a non-sm_100 device yields PCV_ERR_ARCH.
 */
#ifndef PCV_B200_H
#define PCV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCV_ABI_VERSION 3

#define PCV_OK 0
#define PCV_ERR_ARG (-1)
#define PCV_ERR_ARCH (-2)
#define PCV_ERR_CUDA (-3)
#define PCV_ERR_WORKSPACE (-4)
#define PCV_ERR_UNSUPPORTED (-5)

typedef void *pcv_stream_t; /* cudaStream_t */

int pcv_abi_version(void);
const char *pcv_last_error(void);
/* 0 when `device` is compute capability 10.x (B200), PCV_ERR_ARCH otherwise. */
int pcv_device_ok(int device);
/* Number of kernels this library has launched in this process (bench.py's gpu_launches). */
int64_t pcv_launch_count(void);
/* *counter += inc on the stream: advances the device-side Philox row counter between the
 * replays of a captured CUDA graph (see offset_dev below). */
int pcv_counter_add(uint64_t *counter, uint64_t inc, pcv_stream_t stream);

/* ------------------------------------------------------------------ */
/* Item table (the row-L2-normalised catalog; cvae.py:27-33)           */
/* ------------------------------------------------------------------ */
typedef struct pcv_table pcv_table;

/* W: [n_rows, dim] fp32 row-major, 16-byte aligned.  row_offset is the global
 * index of row 0 (vocab-parallel shards, SURVEY §8e); indices returned by
 * pcv_score_select are global (= local + row_offset).  The table is borrowed,
 * not copied: it must outlive the handle.  dim must be a multiple of 4, <= 128.
 * The handle owns the packed images the tensor-core engines stream with TMA: dim 8/16/32/64/128 the pre-swizzled fp32
 * copy (dim * 4 bytes per row), dim 8 with row norms in (0, 1e4) at creation also the f16 image of the f16 filter (32
 * bytes per row), and a device scalar holding max_j |w_j|_2 that the kernels read.  They are derived from W's values:
 * after W changes in place, call pcv_table_refresh (or re-create the handle when W moves or changes shape). */
int pcv_table_create(const float *W, int64_t n_rows, int dim, int64_t row_offset,
                     pcv_table **out);
void pcv_table_destroy(pcv_table *t);
/* W was updated in place (same pointer, n_rows and dim, e.g. by an optimizer step): re-derive on `stream` everything
 * the handle derived from its values -- max|w|, the pre-swizzled image, the f16 image and the tf32 CE's transposed
 * image when the handle has them (a transposed image not built yet stays lazy).  One pass over W plus a one-thread
 * kernel; no allocation, no synchronisation, no host copy, so it may be captured in a CUDA graph.  Afterwards every
 * entry point gives bit for bit the results of a handle freshly created on the same W.  Whether an f16 image exists
 * stays as decided at creation: if max|w| leaves (0, 1e4) the f16 filter flags every stream for the exact re-scan
 * (exact, slow). */
int pcv_table_refresh(pcv_table *t, pcv_stream_t stream);
/* F.normalize(W, p=2, dim=1, eps=1e-12) row-wise, out-of-place (cvae.py:31,39). */
int pcv_normalize_rows(const float *W, int64_t n_rows, int dim, float *out,
                       pcv_stream_t stream);

/* ------------------------------------------------------------------ */
/* Fused score + select over the catalog                               */
/*   greedy : cvae.py:97-101 (get_recommended_item), pivotcvae.py:191  */
/*   exprace: pivotcvae.py:389-391, parity mode (Exp(1) noise from     */
/*            the caller); throughput: pcv_sigmoid_categorical         */
/* ------------------------------------------------------------------ */
#define PCV_SELECT_GREEDY 0  /* argmax_j <q, w_j>, ties -> lowest j                 */
#define PCV_SELECT_EXPRACE 1 /* argmax_j sigmoid(<q_i, w_j>) / noise[i, j]          */

#define PCV_ENGINE_AUTO 0
#define PCV_ENGINE_SIMT 1    /* exact fp32 FMA chain on CUDA cores                  */
#define PCV_ENGINE_TCGEN05 2 /* tf32 tcgen05 filter + exact fp32 refine (greedy)    */
#define PCV_ENGINE_TCGEN05_F16 3 /* dim 8: f16 tcgen05 filter (f16 accumulators read two per register, packed 16-bit
                                  * maxima) + the same exact fp32 refine: identical results                           */

typedef struct {
  int mode;           /* PCV_SELECT_*                                              */
  int engine;         /* PCV_ENGINE_*                                              */
  const float *noise; /* exprace: [M, n_rows] Exp(1) draws, required; greedy: NULL */
  int no_repeat;      /* 0 (default) = the reference's behaviour: independent per-row arg-max, duplicates inside a slate
                         allowed (cvae.py:97-101; SURVEY F1).  L > 0 (opt-in extension, greedy mode, L <= 16, M % L == 0):
                         rows are the L consecutive slots of M/L slates and slot l takes its best item that slots
                         0..l-1 of the same slate have not taken (pcv_slate_no_repeat runs after the top-1 pass; the
                         workspace must then hold pcv_score_select_workspace_bytes + pcv_score_topk_workspace_bytes).
                         A row shard (row_offset > 0) runs the select without it and then the sharded pair
                         pcv_slate_no_repeat_partials + pcv_slate_no_repeat_merge */
} pcv_select_opts;

/* The workspace must be ZERO-FILLED once when it is allocated (the tcgen05 engine keeps a few
 * counters in it and leaves them zeroed after every call); it may then be reused by any number of
 * calls with the same table and M, one call at a time. */
int pcv_score_select_workspace_bytes(const pcv_table *t, int64_t M, size_t *bytes_host);
/* Q: [M, dim].  out_idx: [M] int64 (global index).  out_val: [M] fp32 (the
 * winning score; for exprace the winning key) or NULL.
 * Non-finite scores (DESIGN.md section 2), every engine alike: +-inf order as numbers and equal ones tie by index,
 * as in torch.max; a NaN score never wins (it counts as -inf; torch.max would return it), and a row with no score
 * above -inf returns its first index (row_offset) with value -inf.  An index is therefore always inside the table.
 * The exponential race keys NaN scores like the oracle's exp does (the clamp maps exp(NaN) to exp(-86)).
 * Workspace: any engine may follow any other on one workspace. */
int pcv_score_select(const pcv_table *t, const float *Q, int64_t M,
                     const pcv_select_opts *opts, int64_t *out_idx, float *out_val,
                     void *workspace, size_t workspace_bytes, pcv_stream_t stream);
/* API-parity path for forward()'s `p` (pivotcvae.py:274, listcvae.py:166):
 * out[M, n_rows] = Q @ W^T, exact fp32 sequential-k FMA chain. */
int pcv_score_logits(const pcv_table *t, const float *Q, int64_t M, float *out,
                     pcv_stream_t stream);
/* Throughput-mode sampled pivot (pivotcvae.py:349-351 and the other *_spi / spt / sgt variants):
 * out_idx[i] ~ Categorical(sigmoid(<q_i, w_j>) / sum_j) over the WHOLE catalog, drawn exactly by rejection
 * (uniform proposal, accept with sigmoid(s_j) / sigmoid(|q_i| max_j|w_j|)): ~2 proposals per row instead of one
 * exponential per (row, item).  Philox4x32-10(seed, row + offset [+ *offset_dev]); every operation is portable
 * IEEE, so the oracle reproduces the draws bit for bit.  The table must be the full catalog (row_offset 0).
 * out_iters (optional): proposals used per row, -1 = inverse-CDF fallback after 1024 rejections.
 * Parity mode (caller-supplied torch noise) is pcv_score_select(PCV_SELECT_EXPRACE, noise). */
int pcv_sigmoid_categorical(const pcv_table *t, const float *Q, int64_t M, uint64_t seed, uint64_t offset,
                            const uint64_t *offset_dev, int64_t *out_idx, int32_t *out_iters,
                            pcv_stream_t stream);
/* Exact top-k over the catalog (torch.topk of the score row; models/deterministic.py:119 in the reference, and the
 * building block of the no-repeat selection): out_idx/out_val [M, k], k <= 16, sorted by score descending, equal
 * scores by ascending index; same fp32 sequential-k FMA chain as pcv_score_select; entries beyond the catalog size
 * are -1 / -inf.  Indices are global (+ row_offset).  Only scores above -inf are listed (a NaN counts as -inf): the
 * rest of the window is -1 / -inf as past the end of a short catalog.  pcv_slate_no_repeat: a slot with no untaken
 * item above -inf keeps its top-1 pick (it may repeat, and it takes nothing from the later slots). */
int pcv_score_topk_workspace_bytes(const pcv_table *t, int64_t M, size_t *bytes_host);
int pcv_score_topk(const pcv_table *t, const float *Q, int64_t M, int k, int64_t *out_idx, float *out_val,
                   void *workspace, size_t workspace_bytes, pcv_stream_t stream);
/* Opt-in no-repeat slate selection (NOT reference behaviour, SURVEY F1; north_star's "already-chosen-item mask").
 * Q: [B*L, dim] slot queries, items: [B*L] the top-1 picks of pcv_score_select (in/out), vals: optional [B*L]
 * winning scores (in/out).  Slates whose picks contain a duplicate are re-selected sequentially: slot l takes its
 * best item (ties -> lowest index) not taken by slots 0..l-1.  Only the rows of those slates are re-scored (exact
 * top-L, one pass).  Workspace: pcv_score_topk_workspace_bytes(t, B*L).  The table must be the whole catalog. */
int pcv_slate_no_repeat(const pcv_table *t, const float *Q, int64_t B, int L, int64_t *items, float *vals,
                        void *workspace, size_t workspace_bytes, pcv_stream_t stream);
/* The same selection on a vocab-parallel catalog: every rank runs the partials on its shard, the caller all-gathers
 * the [B*L, L] keys of the G ranks (one collective), and every rank runs the merge.  Neither call syncs the host or
 * allocates, so both can be captured in a CUDA graph.
 * Shard half.  shard: any row shard (row_offset allowed, n_rows may be < L).  Q: [B*L, dim] slot queries (the whole
 * batch, identical on every rank), items: [B*L] the GLOBAL top-1 picks (identical on every rank, i.e. after the
 * vocab-parallel merge).  For every slate whose picks hold a duplicate, writes this shard's exact top-L of each of its
 * L rows into keys[row * L + e] (e = 0..L-1, best first), as order-preserving int64 keys (the pcv_vp_pack_keys
 * encoding, global index).  Missing entries (shard smaller than L) and all rows of duplicate-free slates hold
 * INT64_MIN.  Workspace: pcv_score_topk_workspace_bytes(shard, B*L). */
int pcv_slate_no_repeat_partials(const pcv_table *shard, const float *Q, int64_t B, int L, const int64_t *items,
                                 int64_t *keys, void *workspace, size_t workspace_bytes, pcv_stream_t stream);
/* keys: [G, B*L, L] the partials of the G shards in shard order (G <= 32).  Re-selects the slates of `items` that hold a
 * duplicate, in place, exactly as pcv_slate_no_repeat does on the whole catalog; vals (optional) gets the winning scores. */
int pcv_slate_no_repeat_merge(const int64_t *keys, int G, int64_t B, int L, int64_t *items, float *vals,
                              pcv_stream_t stream);
/* Vocab-parallel merge (SURVEY §8e) of the per-shard winners of pcv_score_select as ONE all-reduce: keys[i] = int64
 * whose SIGNED maximum over the shards is the winner (largest value, equal values -> lowest global index < 2^32).  The caller runs
 * all_reduce(keys, MAX) (NCCL, int64) between pack and unpack; nothing else crosses NVLink. */
int pcv_vp_pack_keys(const float *vals, const int64_t *idx, int64_t M, int64_t *keys, pcv_stream_t stream);
int pcv_vp_unpack_keys(const int64_t *keys, int64_t M, int64_t *out_idx, float *out_val, pcv_stream_t stream);

/* ------------------------------------------------------------------ */
/* Fused MLP blocks (encoder / prior / PSM / SCM / ListCVAE decoder /  */
/* response MLP): concat+gather+one-hot prologue, Linear+activation    */
/* chain with weights streamed through shared memory, optional         */
/* reparameterisation epilogue.                                        */
/*   pivotcvae.py:159-174,197-240,278-291  listcvae.py:90-132          */
/*   cvae.py:79-92   env/response_model.py:76-87                       */
/* ------------------------------------------------------------------ */
#define PCV_ACT_NONE 0
#define PCV_ACT_LEAKY 1 /* nn.LeakyReLU(0.01) (cvae.py:43)          */
#define PCV_ACT_RELU 2  /* F.relu (env/response_model.py:85)        */

typedef struct {
  const float *W; /* [n_out, n_in] row-major == nn.Linear.weight */
  const float *b; /* [n_out]                                     */
  int n_in, n_out, act;
  /* the same weights pre-tiled by pcv_mlp_pack: required on every layer when the launch runs
   * PCV_MLP_KERNEL_CLUSTER, ignored otherwise.  The caller re-packs after the weights change. */
  const float *Wp;
  /* the same weights split in tf32 hi | lo and pre-swizzled by pcv_mlp_tc_pack: required on every layer when the
   * launch runs PCV_MLP_KERNEL_TC, ignored otherwise. */
  const float *Wt;
} pcv_linear;

#define PCV_SEG_DENSE 0  /* ptr: float[B, width]                                      */
#define PCV_SEG_ONEHOT 1 /* ptr: float r[B, count]; one-hot(sum_l r) of width count+1 */
#define PCV_SEG_GATHER 2 /* ptr: float table[*, width]; idx: int64[B, count] -> count*width floats */

#define PCV_NORM_NONE 0
#define PCV_NORM_SEGMENT 1 /* L2-normalise the whole segment (response_model.py:78)  */

typedef struct {
  int kind;
  const void *ptr;
  const int64_t *idx;
  int width; /* row width (DENSE: segment width; GATHER: table dim)  */
  int count; /* ONEHOT: slate size; GATHER: rows gathered per sample */
  int norm;  /* PCV_NORM_*                                           */
} pcv_segment;

#define PCV_MAX_SEGMENTS 6
#define PCV_MAX_LAYERS 8
#define PCV_MAX_WIDTH 1024 /* widest layer / input supported (hyperparams.py:22,79,91 use 1024-wide response MLPs) */

typedef struct {
  int n_segments;
  pcv_segment seg[PCV_MAX_SEGMENTS];
  int n_layers;
  pcv_linear layer[PCV_MAX_LAYERS];
  /* output: out[b*out_ld + out_col0 + j] = last layer j */
  float *out;
  int out_ld, out_col0;
  /* optional: also copy input segment `copy_seg` (>=0) to out[b*out_ld + 0 ..] —
   * used to place the pivot row at slot 0 of rx (pivotcvae.py:224). */
  int copy_seg;
  /* optional saved tensors for backward (NULL to skip): x0[B, n_in0] is the
   * assembled input, acts[l] is [B, n_out_l] post-activation output of layer l
   * (l < n_layers-1; the last layer's output is `out`). */
  float *x0;
  float *acts[PCV_MAX_LAYERS];
  /* optional reparameterisation epilogue (cvae.py:79-83): the last layer emits
   * [mu | logvar] (2*latent); z[b, j] = eps*exp(0.5*logvar)+mu.  eps from
   * `eps` ([B, latent], parity mode) or Philox(seed, offset) normals. */
  int latent; /* 0 = no reparam */
  const float *eps;
  uint64_t seed, offset;
  float *z;       /* [B, latent] */
  float *eps_out; /* optional [B, latent]: the eps actually used (for backward) */
  const uint64_t *offset_dev; /* optional device counter added to `offset` (CUDA-graph replays) */
} pcv_mlp_desc;

/* Engine policy of a launch (`engine` below). */
#define PCV_MLP_EXACT 0 /* the FFMA engines: sequential-k FMA chain, bit-identical to the CPU oracle */
#define PCV_MLP_TC 1    /* the tensor-core engine when every block of the launch fits it (assembled input <= 64 wide,
                         * layers <= 256 wide, at most one one-hot segment of <= 16 clicks), the FFMA engines otherwise.
                         * tcgen05 3xTF32, activations chained through TMEM: fp32-grade (~1e-6 relative of torch's
                         * addmm) but NOT bit-identical to the FFMA engines */
#define PCV_MLP_AUTO 2  /* PCV_MLP_TC from 2048 batch rows, PCV_MLP_EXACT below */
/* The kernel that runs a launch. */
#define PCV_MLP_KERNEL_TC 0      /* csrc/mlp_tc.cu; reads pcv_linear.Wt */
#define PCV_MLP_KERNEL_CLUSTER 1 /* packed-weight FFMA engine (TMA-fed 4-CTA clusters); reads pcv_linear.Wp */
#define PCV_MLP_KERNEL_STREAM 2  /* streaming FFMA engine; reads W; the only one that writes x0 / acts */

/* *kernel = the kernel that pcv_mlp_fwd (b NULL) or pcv_mlp_fwd2 runs for these descriptors, B and engine.  It reads
 * shapes and saved outputs only, no weight image, launches nothing and needs no GPU: the caller packs the image that
 * kernel reads, then launches with the same arguments. */
int pcv_mlp_plan(const pcv_mlp_desc *a, const pcv_mlp_desc *b, int64_t B, int engine, int *kernel);
/* Runs the kernel pcv_mlp_plan names for the same arguments; PCV_ERR_ARG when a layer lacks the weight image that
 * kernel reads (no fall-back to another engine). */
int pcv_mlp_fwd(const pcv_mlp_desc *d, int64_t B, int engine, pcv_stream_t stream);
/* Two chained blocks in ONE launch: b may read (as DENSE segments) what a writes for the same
 * batch rows, e.g. prior -> reparameterise -> PSM (pivotcvae.py:279-291, 204-210). */
int pcv_mlp_fwd2(const pcv_mlp_desc *a, const pcv_mlp_desc *b, int64_t B, int engine, pcv_stream_t stream);
/* Pre-tile one nn.Linear weight [n_out, n_in] for pcv_linear.Wp: `packed` (device, 128-byte aligned)
 * holds pcv_mlp_packed_bytes(n_in, n_out) bytes. */
size_t pcv_mlp_packed_bytes(int n_in, int n_out);
int pcv_mlp_pack(const float *W, int n_in, int n_out, float *packed, pcv_stream_t stream);
/* The tensor-core engine's image of one nn.Linear weight (pcv_linear.Wt): per 32-k chunk the [n_out_pad16][32] tf32-hi
 * and tf32-lo matrices in the K-major SWIZZLE_128B shared-memory layout, so a chunk is one TMA bulk copy. */
size_t pcv_mlp_tc_packed_bytes(int n_in, int n_out);
int pcv_mlp_tc_pack(const float *W, int n_in, int n_out, float *packed, pcv_stream_t stream);

/* ------------------------------------------------------------------ */
/* Tensor-core GEMMs of the MLP blocks' backward (and forward Linear)  */
/*   train_generative.py:133 loss.backward() through pivotcvae.py:159-174, 204-240: */
/*   the reference runs cuBLAS sgemm + elementwise autograd kernels.   */
/* C[M, N] = A[M, K] . B[N, K]^T ("TN": both operands row-major with K contiguous, fp32, 16-byte aligned, leading */
/* dimensions multiples of 4 floats), tcgen05 kind::tf32 with fp32 accumulation in TMEM, operands fed by TMA tensor */
/* maps (ragged M / N / K are zero-filled by the TMA unit).  With A_lo / B_lo (= x - tf32(x)) three MMAs per k-step */
/* (hi*hi + lo*hi + hi*lo, "3xTF32") give fp32-grade products.                                                     */
/* Epilogue, in this order: + bias[n]; act; * act'(dact_src[m, n]) (derivative taken from a saved post-activation */
/* output); store C (and its tf32 residual C_lo), optional transposed copy Ct [N, M] (+ Ct_lo).  split_k > 1: slice z */
/* (K cut in 32-float blocks) writes raw partial sums to C + z * c_split_stride (pcv_wgrad_reduce adds them up).   */
/* ------------------------------------------------------------------ */
typedef struct {
  const float *A, *A_lo; int64_t lda;
  const float *B, *B_lo; int64_t ldb;
  int64_t M, N, K;
  int split_k;
  float *C; int64_t ldc; int64_t c_split_stride;
  float *C_lo;
  float *Ct, *Ct_lo; int64_t ldct;
  const float *bias;
  int act;
  const float *dact_src; int64_t ld_dact; int dact;
} pcv_gemm_desc;
int pcv_gemm_tn(const pcv_gemm_desc *d, pcv_stream_t stream);
/* Batched transposes (<= 12 per launch): dst[c, r] = src[r, c]; optional dst_lo = tf32 residual of the transposed copy, */
/* optional src_lo [rows, ld_src] = tf32 residual of the source.  Lays out the saved activations / weights of an MLP   */
/* block K-major for the weight-gradient and input-gradient GEMMs.                                                      */
typedef struct {
  const float *src; int64_t ld_src; int rows, cols;
  float *dst; int64_t ld_dst;
  float *dst_lo;
  float *src_lo;
} pcv_transpose_job;
int pcv_transpose_batch(const pcv_transpose_job *jobs, int n_jobs, pcv_stream_t stream);
/* dW[o, i] = sum_z part[z][o][i] in fixed order (deterministic), db[o] = sum_b Gt[o, b] (Gt = transposed output gradient). */
int pcv_wgrad_reduce(const float *part, int n_split, int64_t split_stride, int64_t ld_part, int n_out, int n_in, float *dW,
                     int64_t ld_dw, const float *Gt, int64_t ld_gt, int64_t B, float *db, pcv_stream_t stream);

/* KL(q || p) between diagonal Gaussians, summed over batch and latent
 * (train_generative.py:61) plus analytic grads (any grad pointer may be NULL).
 * kl_out: device scalar (overwritten, not accumulated). */
int pcv_kl_fwd_bwd(const float *mu, const float *logvar, const float *pmu,
                   const float *plogvar, int64_t n, float *kl_out, float *dmu,
                   float *dlogvar, float *dpmu, float *dplogvar, pcv_stream_t stream);

/* ------------------------------------------------------------------ */
/* Fused streaming masked soft-max cross-entropy over the catalog      */
/*   train_generative.py:36-42 (downsample), :59 (CrossEntropyLoss),   */
/*   pivotcvae.py:274 (logits) — logits never reach HBM.               */
/* loss_row[i] = log(sum_{j in mask_i} e^{x_ij} + (N-|mask_i|)) - x_{i,t_i}   */
/* mask_i = {t_i} U Bernoulli(keep_prob) per (i, j); masked-out logits are 0.   */
/* Philox mode draws the mask as a gap process (Geometric(keep) distances inside */
/* 1024-column blocks, integer inverse CDF) and visits only the kept columns:    */
/* O(n_neg) work per row instead of O(N).                                        */
/* (not -inf) exactly as `pred * mask` does (SURVEY F7).               */
/* dq[i,:] = d loss_row[i] / d q_i.  The gradient w.r.t. the table is a  */
/* second pass, pcv_ce_table_grad (fine_tune=True).                    */
/* ------------------------------------------------------------------ */
typedef struct {
  double keep_prob;        /* n_neg / N; >= 1 means full-catalog soft-max, no RNG    */
  const uint32_t *bitmask; /* parity mode: [M, ceil(N/32)] bit j%32 of word j/32 = Bernoulli draw (target is OR-ed in by the kernel) */
  uint64_t seed, offset;   /* Philox mode (bitmask == NULL && keep_prob < 1)         */
  const uint64_t *offset_dev; /* optional device counter added to `offset` (CUDA-graph replays) */
  int engine;              /* PCV_CE_ENGINE_*: EXACT (default) or TF32 (dense mask, dim 8, 16, 32, 64 or 128: logits
                              AND the gradient contraction on the tensor cores, loss ~1e-4 / dq ~1e-3 relative — the
                              reduced-precision tolerance, reproducible bit for bit; other dims return
                              PCV_ERR_UNSUPPORTED).  The first TF32
                              call on a table handle builds its transposed tile image (one-off allocation + device
                              sync, like pcv_table_create): run it once outside any CUDA-graph capture.  The handle
                              keeps that image until it is destroyed (pcv_table_refresh keeps it current): n_rows *
                              dim * 4 bytes (rounded up to whole tiles) at dim >= 16, twice that at dim 8 */
} pcv_ce_mask;
#define PCV_CE_ENGINE_EXACT 0
#define PCV_CE_ENGINE_TF32 1

int pcv_ce_workspace_bytes(const pcv_table *t, int64_t M, size_t *bytes_host);
/* Single streaming pass producing loss rows, log-sum-exp and dq (forward and
 * the gradient in one pass; backward is a scale by the upstream gradient).
 * The table must be the whole catalog (row_offset 0); shards go through pcv_ce_partials. */
int pcv_ce_fwd_bwd(const pcv_table *t, const float *Q, const int64_t *targets,
                   int64_t M, const pcv_ce_mask *mask, float *loss_rows, float *lse,
                   float *dq, void *workspace, size_t workspace_bytes,
                   pcv_stream_t stream);

/* Vocab-parallel CE (SURVEY §8e): the same streaming pass over ONE row shard of the table (pcv_table_create with
 * row_offset), full-catalog soft-max only (keep_prob >= 1; engine EXACT, or TF32 at dim 8 to 128).  rec_out: [M, 2 + dim] per-row
 * partial records {m, l, acc[dim]}: m = max logit over the shard, l = sum_j e^{x_j - m}, acc = sum_j e^{x_j - m} w_j.
 * The caller all-gathers the records of the G shards (ONE collective of M * (2 + dim) floats per rank) and
 * pcv_ce_vp_merge combines them: lse = M' + log sum_g l_g e^{m_g - M'}, loss = lse - <q, w_t>,
 * dq = sum_g acc_g e^{m_g - M'} / L - w_t, with the target row taken from the WHOLE fp32 table W_full [N, dim]
 * (every rank keeps it), exact FMA chain.  Every rank ends up with the full dq, so no further all-reduce is needed. */
int pcv_ce_partials(const pcv_table *shard, const float *Q, const int64_t *targets, int64_t M,
                    const pcv_ce_mask *mask, float *rec_out, void *workspace, size_t workspace_bytes,
                    pcv_stream_t stream);
int pcv_ce_vp_merge(const float *recs, int G, const float *W_full, int dim, const float *Q, const int64_t *targets,
                    int64_t M, float *loss_rows, float *lse, float *dq, pcv_stream_t stream);

/* Candidate-mode (sampled soft-max) CE — the reference's default training mode
 * (train_generative.py:52-56; pivotcvae.py:265-271, listcvae.py:157-163):
 * p[i, c] = <W[candidates[i, c]], q_i>, loss_rows[i] = CE(p[i, :], target_pos[i]).
 * candidates: [M, n_cand] int64 item ids, target_pos: [M] int64 column of the target.
 * dq[i, :] = d loss_rows[i] / d q_i; logits_out (optional) = p [M, n_cand]. */
int pcv_cand_ce_fwd_bwd(const pcv_table *t, const float *Q, const int64_t *candidates,
                        const int64_t *target_pos, int64_t M, int n_cand, float *loss_rows,
                        float *lse, float *dq, float *logits_out, pcv_stream_t stream);

/* Gradient of the catalog CE w.r.t. the item table (fine_tune=True trains docEmbed, cvae.py:27-33):
 *   dW[j] = sum_i row_scale[i] * m_ij * (e^{x_ij - lse_i} - [t_i = j]) * q_i
 * with the forward's mask m (masked-out logits are constant zeros: no gradient).  Q, targets, M and mask are those of
 * the pcv_ce_fwd_bwd call, lse [M] is what it returned, row_scale [M] = d loss / d loss_rows[i] (device).  dW [n_rows,
 * dim] is OVERWRITTEN.  Dims 4..128 as the forward.
 * Row shard (vocab-parallel, pcv_table_create with row_offset > 0; row_offset must be a multiple of 128, else
 * PCV_ERR_ARG): dW holds the shard's n_rows rows only, targets stay global indices (a one-hot term counts only when
 * its target lies in [row_offset, row_offset + n_rows)), and lse must be the WHOLE catalog's (pcv_ce_fwd_bwd on the
 * full table, or pcv_ce_vp_merge).  A bitmask is the shard's own columns: row i holds ceil(n_rows / 32) words, bit j
 * is global column row_offset + j (columns [row_offset / 32, ceil((row_offset + n_rows) / 32)) of the forward's mask).
 * Every row of a shard equals that row of the whole-table result: bit for bit on the tf32 path, and on the exact pass
 * when both plans have one row split.  Paths (the forward's routing):
 *  - bitmask, or keep_prob >= 1 with engine EXACT: item-major exact pass — a CTA owns 128 items and streams every
 *    query row, logits re-derived with the forward's fp32 FMA chain, rows summed in a fixed order (+ a fixed-order
 *    reduce of row splits when the catalog is small).  REPRODUCIBLE bit for bit;
 *  - keep_prob >= 1 with engine TF32 (dims 8..128, else PCV_ERR_UNSUPPORTED): the same item-major sweep on the tensor
 *    cores (tcgen05 kind::tf32: logits S^T = W_slab . Q^T, then dW += P^T . Q with P^T read from tensor memory; dW
 *    stays in TMEM for the whole sweep).  Reduced precision like the tf32 forward (tf32 logits, within 2^-9 |q| |w|;
 *    tf32 products in the contraction), REPRODUCIBLE bit for bit; needs no workspace beyond the query;
 *  - Philox (keep_prob < 1, no bitmask): regenerates exactly the forward's gap-process mask from seed, offset and
 *    *offset_dev, O(M * n_neg) work (a shard walks only the 1024-column blocks it overlaps: O(M * n_neg * n_rows / N)),
 *    float atomics: NOT reproducible bit for bit (last-bit differences run to run).
 * Workspace: pcv_ce_table_grad_workspace_bytes for the same table, M and mask (no zero-fill needed).  No allocation,
 * no host sync. */
int pcv_ce_table_grad_workspace_bytes(const pcv_table *t, int64_t M, const pcv_ce_mask *mask, size_t *bytes_host);
int pcv_ce_table_grad(const pcv_table *t, const float *Q, const int64_t *targets, int64_t M,
                      const pcv_ce_mask *mask, const float *lse, const float *row_scale,
                      float *dW, void *workspace, size_t workspace_bytes, pcv_stream_t stream);
/* Candidate mode: dW[candidates[i, c]] += row_scale[i] * (softmax_c(p[i, :]) - [c = target_pos[i]]) * q_i for every
 * column c (a duplicate candidate once per occurrence), logits re-derived from lse (of pcv_cand_ce_fwd_bwd).  ADDS
 * into dW: the caller zero-fills it.  Float atomics: not reproducible bit for bit.  A row shard (row_offset a multiple
 * of 128, else PCV_ERR_ARG) takes the whole catalog's lse and global candidate ids; it skips candidates outside it and
 * adds into dW[j - row_offset] ([n_rows, dim]). */
int pcv_cand_ce_table_grad(const pcv_table *t, const float *Q, const int64_t *candidates, const int64_t *target_pos,
                           int64_t M, int n_cand, const float *lse, const float *row_scale, float *dW, pcv_stream_t stream);

/* ------------------------------------------------------------------ */
/* Simulator response models, gather-plus-dot (env/response_model.py)  */
/*   URM      :129-150   URM_P :286-295   URM_P_MR :315-323            */
/* ------------------------------------------------------------------ */
#define PCV_URM 0
#define PCV_URM_P 1
#define PCV_URM_P_MR 2

typedef struct {
  int variant;
  const float *doc_table;  /* [I, D] raw (un-normalised) item embeddings      */
  const float *user_table; /* [U, D] raw user embeddings (used un-normalised, response_model.py:145) */
  const float *item_bias;  /* [I]                                             */
  const float *user_bias;  /* [U]                                             */
  const float *pos_bias;   /* [L]       (URM_P*)                              */
  const float *pos_dep;    /* [L*D] flat, read as a (D, L) view (response_model.py:292) */
  float mr_factor;         /* URM_P_MR                                        */
  int L, D;
} pcv_urm_desc;

/* out: [B, L] final score (URM: sigmoid(raw); URM_P: sigmoid(raw)+pos terms; ...). */
int pcv_urm_fwd(const pcv_urm_desc *d, const int64_t *slates, const int64_t *users,
                int64_t B, float *out, pcv_stream_t stream);

/* ------------------------------------------------------------------ */
/* Response-model pre-training (SURVEY 8f N4: pretrain_env.py:25-139):  */
/* the embeddings are trainable there, so the gather + normalise prologue */
/* of env/response_model.py:76-83 needs a backward.                      */
/* ------------------------------------------------------------------ */
/* x0[b, :] = [ normalize(concat_l doc[slates[b, l]]) | normalize(usr[users[b]]) ] (usr NULL = no_user); x0 is
 * [B, ld], inv_norm [B, 2] keeps 1 / max(|raw|, 1e-12) of both segments for the backward. */
int pcv_gather_norm_fwd(const float *doc, const float *usr, const int64_t *slates, const int64_t *users, int64_t B, int L,
                        int D, float *x0, int64_t ld, float *inv_norm, pcv_stream_t stream);
/* d_doc / d_usr (zero-initialised by the caller, same shapes as the tables) += the gradient of x0 w.r.t. the raw rows. */
int pcv_gather_norm_bwd(const float *g, int64_t ldg, const float *x0, int64_t ld, const float *inv_norm, const int64_t *slates,
                        const int64_t *users, int64_t B, int L, int D, float *d_doc, float *d_usr, pcv_stream_t stream);
/* Backward of the reparameterisation (cvae.py:79-83) folded into the gradient of a block's [mu | logvar] output
 * (out: [B, ld_out] the block's saved output, columns 0..2Z-1; d_out / d_z may be NULL): g [B, 2Z] contiguous. */
int pcv_reparam_bwd(const float *d_out, int64_t ld_dout, const float *d_z, const float *eps, const float *out, int64_t ld_out,
                    int64_t B, int Z, float *g, pcv_stream_t stream);
/* nn.BCELoss()(sigmoid(pred), target) (pretrain_env.py:57-58,84; logs clamped at -100) and dpred (optional). */
int pcv_bce_sigmoid(const float *pred, const float *target, int64_t n, float *loss, float *dpred, pcv_stream_t stream);

/* ------------------------------------------------------------------ */
/* Slate metrics of the variation-control evaluation (analysis.py:5-30) */
/* ------------------------------------------------------------------ */
/* ils[b] = (sum_{i,j} cos(e_i, e_j) - L) / (L (L-1)) over the L items of slate b (get_ILS);
 * bitmap (optional, ceil(N/32) words, zeroed by the caller) gets bit `item` set for every
 * recommended item; pcv_popcount(bitmap) / N is get_coverage. table: [N, D] raw embeddings. */
int pcv_slate_metrics(const float *table, int D, const int64_t *slates, int64_t B, int L, float *ils,
                      uint32_t *bitmap, pcv_stream_t stream);
int pcv_popcount(const uint32_t *bitmap, int64_t words, uint64_t *count, pcv_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PCV_B200_H */
