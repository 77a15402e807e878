/*
 * pcv_oracle.c — CPU restatement of the PivotCVAE slate-generation hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under pivotcvae_b200/ may import, link or
 * call this file; only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference leg use it, and only as the checker / the
 * CPU baseline.  The product path is libpcv_b200.so and has no CPU fallback.
 *
 * Parity pinning: the reference ships no tests or golden vectors (SURVEY §4),
 * so this oracle is pinned against outputs of the reference's own Python
 * classes, generated in the build container by tests/golden/make_golden.py
 * (importing /root/reference) and committed under tests/golden/ (npz files);
 * tests/test_oracle_golden.py checks every function here against them.
 * Philox4x32-10 is pinned against the Random123 known-answer vectors.
 *
 * Arithmetic: plain C, fp32, every fused multiply-add is an explicit fmaf()
 * (build with -ffp-contract=off), K loops are sequential and ascending — the
 * order SURVEY F3 shows the reference's torch.mm has at D=8.
 * Each function cites the reference file:line it follows (/root/reference).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <pthread.h>
#include <stdatomic.h>

/* ---- minimal pthread parallel-for (libgomp is not in the image) ---- */
typedef void (*orc_body)(int64_t begin, int64_t end, void *ctx);
static int g_threads = 1;
void orc_set_threads(int n) { g_threads = n < 1 ? 1 : (n > 256 ? 256 : n); }
int orc_get_threads(void) { return g_threads; }
typedef struct {
  atomic_llong next;
  int64_t n, grain;
  orc_body f;
  void *ctx;
} orc_pf;
static void *orc_pf_worker(void *p) {
  orc_pf *w = (orc_pf *)p;
  for (;;) {
    int64_t b = atomic_fetch_add(&w->next, w->grain);
    if (b >= w->n) break;
    int64_t e = b + w->grain > w->n ? w->n : b + w->grain;
    w->f(b, e, w->ctx);
  }
  return NULL;
}
static void parallel_for(int64_t n, int64_t grain, orc_body f, void *ctx) {
  int64_t chunks = (n + grain - 1) / grain;
  int nt = (int)(chunks < g_threads ? chunks : g_threads);
  if (nt <= 1) { f(0, n, ctx); return; }
  orc_pf w;
  atomic_init(&w.next, 0);
  w.n = n; w.grain = grain; w.f = f; w.ctx = ctx;
  pthread_t th[256];
  for (int t = 1; t < nt; ++t) pthread_create(&th[t], NULL, orc_pf_worker, &w);
  orc_pf_worker(&w);
  for (int t = 1; t < nt; ++t) pthread_join(th[t], NULL);
}

#define ORC_ACT_NONE 0
#define ORC_ACT_LEAKY 1
#define ORC_ACT_RELU 2

/* ---- portable exp: same IEEE op sequence as pcv_expf in the CUDA library ---- */
static inline float orc_expf_(float x) {
  x = fminf(fmaxf(x, -86.0f), 88.0f);
  const float magic = 12582912.0f;
  float t = fmaf(x, 1.44269504088896341f, magic);
  float n = t - magic;
  float r = fmaf(n, -0.693145751953125f, x);
  r = fmaf(n, -1.42860682030941723212e-6f, r);
  float p = 1.9875691500e-4f;
  p = fmaf(p, r, 1.3981999507e-3f);
  p = fmaf(p, r, 8.3334519073e-3f);
  p = fmaf(p, r, 4.1665795894e-2f);
  p = fmaf(p, r, 1.6666665459e-1f);
  p = fmaf(p, r, 5.0000001201e-1f);
  float r2 = r * r;
  float e = fmaf(p, r2, r) + 1.0f;
  int ni = (int)n;
  union { uint32_t u; float f; } s;
  s.u = (uint32_t)(ni + 127) << 23;
  return e * s.f;
}

void orc_expf(const float *x, int64_t n, float *y) {
  for (int64_t i = 0; i < n; ++i) y[i] = orc_expf_(x[i]);
}

/* ---- Philox4x32-10 (Salmon et al. SC'11; Random123 philox.h) ---- */
void orc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

/* Bernoulli(keep_prob) bitmask of the CE Philox mode (train_generative.py:39), bit (j & 31) of
 * word j >> 5.  The library draws it as a gap process: inside every block of 1024 consecutive
 * columns the distance to the next kept column is Geometric(keep) (memoryless => the columns are
 * i.i.d. Bernoulli(keep)).  Gap = #{g in 1..1024 : u < T[g]}, T[g] = floor(T[g-1] * q32 / 2^32),
 * T[0] = 2^32, q32 = round((1-keep) * 2^32); u = Philox word k&3 of call
 * (block, row+offset lo, hi, 3 + 16*(k>>2)). */
void orc_bernoulli_bitmask(uint64_t seed, uint64_t offset, int64_t M, int64_t N, double keep_prob,
                           uint32_t *bits) {
  enum { GB = 1024 };
  static uint32_t T[GB + 1];
  double qd = (1.0 - keep_prob) * 4294967296.0;
  uint32_t q32 = qd <= 0.0 ? 0u : (qd >= 4294967295.0 ? 0xffffffffu : (uint32_t)(qd + 0.5));
  uint64_t t = 0x100000000ull;
  T[0] = 0xffffffffu;
  for (int g = 1; g <= GB; ++g) { t = (t * (uint64_t)q32) >> 32; T[g] = (uint32_t)t; }
  int64_t words = (N + 31) / 32;
  memset(bits, 0, (size_t)(M * words) * sizeof(uint32_t));
  uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
  int64_t n_blocks = (N + GB - 1) / GB;
  for (int64_t i = 0; i < M; ++i) {
    uint64_t r = (uint64_t)i + offset;
    for (int64_t b = 0; b < n_blocks; ++b) {
      int c = -1;
      uint32_t o[4] = {0, 0, 0, 0};
      for (int k = 0;; ++k) {
        if ((k & 3) == 0) {
          uint32_t ctr[4] = {(uint32_t)b, (uint32_t)r, (uint32_t)(r >> 32), 3u + ((uint32_t)(k >> 2) << 4)};
          orc_philox4x32_10(ctr, key, o);
        }
        uint32_t u = o[k & 3];
        int gap = 0;
        for (int g = 1; g <= GB; ++g) { if (u < T[g]) gap = g; else break; }
        c += 1 + gap;
        if (c >= GB) break;
        int64_t j = b * GB + c;
        if (j >= N) break;
        bits[i * words + (j >> 5)] |= 1u << (j & 31);
      }
    }
  }
}

/* ---- cvae.py:31,39  F.normalize(W, p=2, dim=1) with eps 1e-12 ---- */
void orc_normalize_rows(const float *W, int64_t n, int dim, float *out) {
  for (int64_t i = 0; i < n; ++i) {
    float ss = 0.f;
    for (int k = 0; k < dim; ++k) ss = fmaf(W[i * dim + k], W[i * dim + k], ss);
    float nrm = fmaxf(sqrtf(ss), 1e-12f);
    for (int k = 0; k < dim; ++k) out[i * dim + k] = W[i * dim + k] / nrm;
  }
}

/* ---- cvae.py:85-92  get_condition: one-hot of the click count ---- */
void orc_condition(const float *r, int64_t B, int L, float *cond) {
  for (int64_t b = 0; b < B; ++b) {
    float s = 0.f;
    for (int l = 0; l < L; ++l) s += r[b * L + l];
    int hot = (int)s;
    for (int e = 0; e <= L; ++e) cond[b * (L + 1) + e] = (e == hot) ? 1.f : 0.f;
  }
}

/* ---- nn.Linear + activation (pivotcvae.py:170-173, 208-210, 218-220, 236-239;
 *      listcvae.py:100-103, 116-118; env/response_model.py:84-86) ---- */
typedef struct { const float *x; int K; const float *Wt, *b; int N, act; float *y; } lin_ctx;
static void lin_body(int64_t i0, int64_t i1, void *p) {
  lin_ctx *c = (lin_ctx *)p;
  const int N = c->N, K = c->K;
  float acc[1024];
  for (int64_t i = i0; i < i1; ++i) {
    const float *xi = c->x + i * K;
    for (int n = 0; n < N; ++n) acc[n] = 0.f;
    /* per output n: acc = fmaf(x[k], W[n][k], acc), k ascending (vectorised over n) */
    for (int k = 0; k < K; ++k) {
      const float xk = xi[k];
      const float *w = c->Wt + (int64_t)k * N;
      for (int n = 0; n < N; ++n) acc[n] = fmaf(xk, w[n], acc[n]);
    }
    for (int n = 0; n < N; ++n) {
      float v = acc[n] + c->b[n];
      if (c->act == ORC_ACT_LEAKY) v = v > 0.f ? v : 0.01f * v; /* nn.LeakyReLU() default slope, cvae.py:43 */
      else if (c->act == ORC_ACT_RELU) v = v > 0.f ? v : 0.f;
      c->y[i * N + n] = v;
    }
  }
}
/* W: [N, K] row-major (nn.Linear.weight); N <= 1024 */
void orc_linear(const float *x, int64_t B, int K, const float *W, const float *b, int N, int act,
                float *y) {
  float *Wt = (float *)malloc((size_t)N * K * sizeof(float));
  for (int n = 0; n < N; ++n)
    for (int k = 0; k < K; ++k) Wt[(int64_t)k * N + n] = W[(int64_t)n * K + k];
  lin_ctx c = {x, K, Wt, b, N, act, y};
  parallel_for(B, 16, lin_body, &c);
  free(Wt);
}

/* ---- cvae.py:79-83  reparametrize: std = exp(0.5*logvar); z = eps*std + mu ---- */
void orc_reparam(const float *mu, const float *logvar, const float *eps, int64_t n, float *z) {
  for (int64_t i = 0; i < n; ++i) {
    float sd = orc_expf_(logvar[i] * 0.5f);
    float t = eps[i] * sd;
    z[i] = t + mu[i];
  }
}

/* ---- cvae.py:97-101 get_recommended_item / pivotcvae.py:191 pick_pivot (greedy),
 *      pivotcvae.py:349-351 etc. (sampled): Categorical(sigmoid(s)).sample() is
 *      argmax_j p_j / E_j, E ~ Exp(1) (torch multinomial fast path) which equals
 *      argmin_j E_j * (1 + exp(-s_j)); out_val = -T (larger is better).
 * mode 0 greedy, 1 exponential race with noise[M,N].  Ties -> lowest index. ---- */
#define ORC_JB 256
#define ORC_RB 8
typedef struct {
  const float *Wt, *Q, *noise; int64_t N, M; int D, mode; int64_t *out_idx; float *out_val;
} ss_ctx;
static void ss_body(int64_t rb0, int64_t rb1, void *p) {
  ss_ctx *c = (ss_ctx *)p;
  const int64_t N = c->N, M = c->M;
  const int D = c->D;
  for (int64_t rb = rb0; rb < rb1; ++rb) {
    int64_t i0 = rb * ORC_RB, i1 = i0 + ORC_RB > M ? M : i0 + ORC_RB;
    float best[ORC_RB];
    int64_t bidx[ORC_RB];
    for (int r = 0; r < ORC_RB; ++r) { best[r] = -INFINITY; bidx[r] = 0; }
    float s[ORC_JB];
    for (int64_t j0 = 0; j0 < N; j0 += ORC_JB) {
      int jn = (int)(N - j0 < ORC_JB ? N - j0 : ORC_JB);
      for (int64_t i = i0; i < i1; ++i) {
        const float *q = c->Q + i * D;
        for (int jj = 0; jj < jn; ++jj) s[jj] = 0.f;
        for (int k = 0; k < D; ++k) {
          const float qk = q[k];
          const float *w = c->Wt + (int64_t)k * N + j0;
          for (int jj = 0; jj < jn; ++jj) s[jj] = fmaf(qk, w[jj], s[jj]);
        }
        if (c->mode == 1) {
          const float *e = c->noise + i * N + j0;
          for (int jj = 0; jj < jn; ++jj) {
            float t = 1.0f + orc_expf_(-s[jj]);
            s[jj] = -(e[jj] * t);
          }
        }
        float b = best[i - i0];
        int64_t bi = bidx[i - i0];
        for (int jj = 0; jj < jn; ++jj)
          if (s[jj] > b) { b = s[jj]; bi = j0 + jj; }
        best[i - i0] = b;
        bidx[i - i0] = bi;
      }
    }
    for (int64_t i = i0; i < i1; ++i) {
      c->out_idx[i] = bidx[i - i0];
      if (c->out_val) c->out_val[i] = best[i - i0];
    }
  }
}
void orc_score_select(const float *W, int64_t N, int D, const float *Q, int64_t M, int mode,
                      const float *noise, int64_t *out_idx, float *out_val) {
  float *Wt = (float *)malloc((size_t)N * D * sizeof(float));
  for (int64_t j = 0; j < N; ++j)
    for (int k = 0; k < D; ++k) Wt[(int64_t)k * N + j] = W[j * D + k];
  ss_ctx c = {Wt, Q, noise, N, M, D, mode, out_idx, out_val};
  parallel_for((M + ORC_RB - 1) / ORC_RB, 1, ss_body, &c);
  free(Wt);
}

/* ---- pivotcvae.py:349-351 (and the other sampled variants): samp = Categorical(sigmoid(scores)).sample()
 *      in throughput mode: exact rejection sampling, restating pivotcvae_b200/csrc/sampler.cu operation by
 *      operation (Philox proposal `it` of row r -> (x, y, z, w); j = hi64((x:y) * N), void when
 *      lo64 < 2^64 mod N; accept iff z < (u64)(min(sigmoid(s_j) / sigma_b, 1) * 2^32);
 *      sigma_b = sigmoid(|q| * max_j|w_j| * 1.0001 + 1e-6); after 1024 proposals: inverse CDF in double). ---- */
static inline float orc_sigmoidf_(float x) { return 1.0f / (1.0f + orc_expf_(-x)); }
static inline float orc_chain_(const float *q, const float *w, int D) {
  float s = 0.f;
  for (int k = 0; k < D; ++k) s = fmaf(q[k], w[k], s);
  return s;
}
void orc_sigmoid_categorical(const float *W, int64_t N, int D, const float *Q, int64_t M, uint64_t seed,
                             uint64_t offset, int64_t *out_idx, int32_t *out_iters) {
  float m2 = 0.f;
  for (int64_t j = 0; j < N; ++j) {
    float ss = orc_chain_(W + j * D, W + j * D, D);
    if (ss > m2) m2 = ss;
  }
  const float max_row_norm = sqrtf(m2) * 1.000001f;   /* pcv_table_create */
  const uint64_t lemire_t = (0ull - (uint64_t)N) % (uint64_t)N;
  for (int64_t i = 0; i < M; ++i) {
    const float *q = Q + i * D;
    const float sigma_b = orc_sigmoidf_(sqrtf(orc_chain_(q, q, D)) * max_row_norm * 1.0001f + 1e-6f);
    const uint64_t r = (uint64_t)i + offset;
    int64_t pick = -1;
    uint32_t w0 = 0;
    for (int it = 0; it < 1024 && pick < 0; ++it) {
      uint32_t ctr[4] = {(uint32_t)it, (uint32_t)r, (uint32_t)(r >> 32), 4u};
      uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
      uint32_t o[4];
      orc_philox4x32_10(ctr, key, o);
      if (it == 0) w0 = o[3];
      const uint64_t u = ((uint64_t)o[0] << 32) | o[1];
      const unsigned __int128 m = (unsigned __int128)u * (uint64_t)N;
      const int64_t j = (int64_t)(uint64_t)(m >> 64);
      if ((uint64_t)m < lemire_t) continue;
      const float ratio = fminf(orc_sigmoidf_(orc_chain_(q, W + j * D, D)) / sigma_b, 1.0f);
      const uint64_t thr = (uint64_t)(ratio * 4294967296.0f);
      if ((uint64_t)o[2] < thr) {
        pick = j;
        if (out_iters) out_iters[i] = it + 1;
      }
    }
    if (pick < 0) {
      double total = 0.0;
      for (int64_t j = 0; j < N; ++j) total += (double)orc_sigmoidf_(orc_chain_(q, W + j * D, D));
      const double target = ((double)w0 + 0.5) * (1.0 / 4294967296.0) * total;
      double acc = 0.0;
      pick = N - 1;
      for (int64_t j = 0; j < N; ++j) {
        acc += (double)orc_sigmoidf_(orc_chain_(q, W + j * D, D));
        if (acc >= target) { pick = j; break; }
      }
      if (out_iters) out_iters[i] = -1;
    }
    out_idx[i] = pick;
  }
}

/* ---- pivotcvae.py:274 / listcvae.py:166  p = mm(prox_emb, table.t()) ---- */
void orc_score_logits(const float *W, int64_t N, int D, const float *Q, int64_t M, float *out) {
  for (int64_t i = 0; i < M; ++i)
    for (int64_t j = 0; j < N; ++j) {
      float s = 0.f;
      for (int k = 0; k < D; ++k) s = fmaf(Q[i * D + k], W[j * D + k], s);
      out[i * N + j] = s;
    }
}

/* ---- train_generative.py:36-42 downsample + :59 CrossEntropyLoss, and its
 * gradient w.r.t. the query rows (table frozen, cvae.py:32).
 * bitmask: Bernoulli draws [M, ceil(N/32)] or NULL (= keep everything).
 * mask_i = {t_i} U draws; masked-out logits are 0 (pred * mask).
 * loss_rows[i] = logsumexp_j(y_ij) - y_{i,t_i};  dq = d loss_rows[i] / d q_i. ---- */
typedef struct {
  const float *W, *Q; int64_t N; int D; const int64_t *targets; const uint32_t *bitmask;
  float *loss_rows, *lse_out, *dq;
} ce_ctx;
static void ce_body(int64_t r0, int64_t r1, void *p) {
  ce_ctx *c = (ce_ctx *)p;
  const int64_t N = c->N;
  const int D = c->D;
  const float *W = c->W;
  const uint32_t *bitmask = c->bitmask;
  int64_t words = (N + 31) / 32;
  for (int64_t i = r0; i < r1; ++i) {
    const float *q = c->Q + i * D;
    int64_t t = c->targets[i];
    /* pass 1: max of masked logits */
    float mx = -INFINITY;
    for (int64_t j = 0; j < N; ++j) {
      int in = bitmask ? (int)((bitmask[i * words + (j >> 5)] >> (j & 31)) & 1u) : 1;
      if (j == t) in = 1;
      float y = 0.f;
      if (in) {
        float s = 0.f;
        for (int k = 0; k < D; ++k) s = fmaf(q[k], W[j * D + k], s);
        y = s;
      }
      if (y > mx) mx = y;
    }
    double L = 0.0;
    double acc[128];
    for (int k = 0; k < D; ++k) acc[k] = 0.0;
    float yt = 0.f;
    for (int64_t j = 0; j < N; ++j) {
      int in = bitmask ? (int)((bitmask[i * words + (j >> 5)] >> (j & 31)) & 1u) : 1;
      if (j == t) in = 1;
      float y = 0.f;
      if (in) {
        float s = 0.f;
        for (int k = 0; k < D; ++k) s = fmaf(q[k], W[j * D + k], s);
        y = s;
      }
      if (j == t) yt = y;
      double pr = exp((double)y - (double)mx);
      L += pr;
      if (in)
        for (int k = 0; k < D; ++k) acc[k] += pr * (double)W[j * D + k];
    }
    double lse = (double)mx + log(L);
    if (c->loss_rows) c->loss_rows[i] = (float)(lse - (double)yt);
    if (c->lse_out) c->lse_out[i] = (float)lse;
    if (c->dq)
      for (int k = 0; k < D; ++k) c->dq[i * D + k] = (float)(acc[k] / L - (double)W[t * D + k]);
  }
}
void orc_ce(const float *W, int64_t N, int D, const float *Q, const int64_t *targets, int64_t M,
            const uint32_t *bitmask, float *loss_rows, float *lse_out, float *dq) {
  ce_ctx c = {W, Q, N, D, targets, bitmask, loss_rows, lse_out, dq};
  parallel_for(M, 4, ce_body, &c);
}

/* ---- candidate-mode CE: train_generative.py:52-56 with p = bmm(docEmbed(candidates), prox)
 * (pivotcvae.py:265-271).  cand: [M, nC] item ids, tpos: [M] target column. ---- */
void orc_cand_ce(const float *W, int D, const float *Q, const int64_t *cand, const int64_t *tpos, int64_t M, int nC,
                 float *loss_rows, float *dq, float *logits) {
  for (int64_t i = 0; i < M; ++i) {
    const float *q = Q + i * D;
    float mx = -INFINITY;
    for (int c = 0; c < nC; ++c) {
      const float *w = W + cand[i * nC + c] * D;
      float s = 0.f;
      for (int k = 0; k < D; ++k) s = fmaf(w[k], q[k], s);
      if (logits) logits[i * nC + c] = s;
      if (s > mx) mx = s;
    }
    double L = 0.0, acc[128];
    for (int k = 0; k < D; ++k) acc[k] = 0.0;
    float st = 0.f;
    for (int c = 0; c < nC; ++c) {
      const float *w = W + cand[i * nC + c] * D;
      float s = 0.f;
      for (int k = 0; k < D; ++k) s = fmaf(w[k], q[k], s);
      if (c == tpos[i]) st = s;
      double pr = exp((double)s - (double)mx);
      L += pr;
      for (int k = 0; k < D; ++k) acc[k] += pr * (double)w[k];
    }
    if (loss_rows) loss_rows[i] = (float)((double)mx + log(L) - (double)st);
    if (dq) {
      const float *wt = W + cand[i * nC + tpos[i]] * D;
      for (int k = 0; k < D; ++k) dq[i * D + k] = (float)(acc[k] / L - (double)wt[k]);
    }
  }
}

/* ---- train_generative.py:61  KLD = -0.5 * sum(1 + lv - plv - (exp(lv) + (mu-pmu)^2)/exp(plv)) ---- */
double orc_kl(const float *mu, const float *lv, const float *pmu, const float *plv, int64_t n,
              float *dmu, float *dlv, float *dpmu, float *dplv) {
  double acc = 0.0;
  for (int64_t i = 0; i < n; ++i) {
    double ev = exp((double)lv[i]), ipv = exp(-(double)plv[i]), dm = (double)mu[i] - (double)pmu[i];
    double ratio = (ev + dm * dm) * ipv;
    acc += 1.0 + (double)lv[i] - (double)plv[i] - ratio;
    if (dmu) dmu[i] = (float)(dm * ipv);
    if (dlv) dlv[i] = (float)(-0.5 * (1.0 - ev * ipv));
    if (dpmu) dpmu[i] = (float)(-dm * ipv);
    if (dplv) dplv[i] = (float)(-0.5 * (ratio - 1.0));
  }
  return -0.5 * acc;
}

/* ---- env/response_model.py:129-150 (URM), :286-295 (URM_P), :315-323 (URM_P_MR).
 * variant 0/1/2.  Quirks kept: raw user row (:145), posDependentBias.view(D, L)
 * (:292), positional terms added after the sigmoid (:294). ---- */
void orc_urm(int variant, const float *doc, const float *usr, const float *ibias,
             const float *ubias, const float *pos_bias, const float *pos_dep, float mr_factor,
             int L, int D, const int64_t *slates, const int64_t *users, int64_t B, float *out) {
  for (int64_t b = 0; b < B; ++b) {
    int64_t u = users[b];
    const float *ue = usr + u * D;
    float de[16][128];
    float mean[128];
    for (int k = 0; k < D; ++k) mean[k] = 0.f;
    for (int l = 0; l < L; ++l) {
      int64_t it = slates[b * L + l];
      const float *d = doc + it * D;
      float ss = 0.f;
      for (int k = 0; k < D; ++k) ss = fmaf(d[k], d[k], ss);
      float nrm = fmaxf(sqrtf(ss), 1e-12f);
      float dot = 0.f;
      for (int k = 0; k < D; ++k) {
        de[l][k] = d[k] / nrm;
        dot = fmaf(de[l][k], ue[k], dot);
        mean[k] += de[l][k];
      }
      float v = dot + ibias[it];
      v = v + ubias[u];
      out[b * L + l] = 1.0f / (1.0f + expf(-v));
    }
    if (variant >= 1) {
      for (int l = 0; l < L; ++l) {
        float pb = 0.f;
        for (int k = 0; k < D; ++k) pb = fmaf(ue[k], pos_dep[k * L + l], pb);
        pb = pb + pos_bias[l];
        out[b * L + l] = out[b * L + l] + pb;
      }
    }
    if (variant == 2) {
      float att[128];
      for (int k = 0; k < D; ++k) att[k] = 1.0f / (1.0f + expf(-(mean[k] / (float)L)));
      for (int l = 0; l < L; ++l) {
        float rel = 0.f;
        for (int k = 0; k < D; ++k) rel = fmaf(de[l][k], att[k], rel);
        out[b * L + l] = out[b * L + l] + rel * mr_factor;
      }
    }
  }
}

/* ---- env/response_model.py:76-83: gather L item rows, L2-normalise the WHOLE
 * flattened (L*D) vector, append the normalised user row. x: [B, L*D (+D)] ---- */
void orc_resp_input(const float *doc, const float *usr, int L, int D, const int64_t *slates,
                    const int64_t *users, int64_t B, int no_user, float *x) {
  int w = L * D + (no_user ? 0 : D);
  for (int64_t b = 0; b < B; ++b) {
    float *xb = x + b * w;
    float ss = 0.f;
    for (int l = 0; l < L; ++l)
      for (int k = 0; k < D; ++k) {
        float v = doc[slates[b * L + l] * D + k];
        xb[l * D + k] = v;
        ss = fmaf(v, v, ss);
      }
    float nrm = fmaxf(sqrtf(ss), 1e-12f);
    for (int e = 0; e < L * D; ++e) xb[e] = xb[e] / nrm;
    if (!no_user) {
      const float *ue = usr + users[b] * D;
      float s2 = 0.f;
      for (int k = 0; k < D; ++k) s2 = fmaf(ue[k], ue[k], s2);
      float n2 = fmaxf(sqrtf(s2), 1e-12f);
      for (int k = 0; k < D; ++k) xb[L * D + k] = ue[k] / n2;
    }
  }
}

/* ---- analysis.py:13-30 get_ILS: normalise the L gathered rows, bmm(emb, emb^T), (sum - L) / (L (L-1)) ---- */
void orc_ils(const float *table, int D, const int64_t *slates, int64_t B, int L, float *ils) {
  for (int64_t b = 0; b < B; ++b) {
    float e[16][128];
    for (int l = 0; l < L; ++l) {
      const float *r = table + slates[b * L + l] * D;
      float ss = 0.f;
      for (int k = 0; k < D; ++k) ss = fmaf(r[k], r[k], ss);
      float nrm = fmaxf(sqrtf(ss), 1e-12f);
      for (int k = 0; k < D; ++k) e[l][k] = r[k] / nrm;
    }
    double tot = 0.0;
    for (int i = 0; i < L; ++i)
      for (int j = 0; j < L; ++j) {
        double d = 0.0;
        for (int k = 0; k < D; ++k) d += (double)e[i][k] * (double)e[j][k];
        tot += d;
      }
    ils[b] = (float)((tot - (double)L) / (double)(L * (L - 1)));
  }
}
