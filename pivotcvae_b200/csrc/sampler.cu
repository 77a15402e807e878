// sampler.cu — exact draw from Categorical(sigmoid(<q, w_j>)) over the whole catalog in O(1) per row.
//
// Replaces pivotcvae.py:349-351, 371-373, 389-391, 409-411, 429-431, 447-454:
//     p = sigmoid(mm(pivot_output, table.t()));  samp = Categorical(p).sample()
// The reference materialises the (B, N) probabilities and torch draws one exponential per (row, item)
// (SURVEY F4).  When the caller supplies that noise (parity mode, identical RNG stream) the race kernel of
// score_select.cu reproduces torch's pick bit for bit.  In throughput mode the noise is ours to choose, and the
// SAME distribution is sampled exactly by rejection:
//
//     repeat:  j ~ Uniform{0..N-1},  accept with probability sigmoid(s_j) / sigma_b
//
// where sigma_b = sigmoid(|q| * max_j |w_j|) >= sigmoid(s_j) for every j (Cauchy-Schwarz; max_j |w_j| is kept
// by the table handle).  P(return j) is proportional to sigmoid(s_j): exactly Categorical(p / sum p).  Scores
// are centred (table rows are unit vectors spread over the sphere), so the acceptance rate is about
// 0.5 / sigma_b: ~2 proposals per row instead of N exponentials — the sampled pivot costs microseconds instead
// of 10 ms at N = 1 M (profiles/r2a_bench.json: 10.3 ms of a 12.1 ms step before this kernel).
//
// Everything is portable IEEE arithmetic (Philox4x32-10, sequential-k FMA chain, pcv_sigmoidf, one division), so
// the oracle restates the sampler bit for bit (oracle/pcv_oracle.c: orc_sigmoid_categorical).
//   proposal it of row r: Philox(ctr = (it, r_lo, r_hi, PCV_STREAM_REJECT), key = seed) -> words (x, y, z, w);
//     u64 = x:y;  j = hi64(u64 * N);  the proposal is void when lo64(u64 * N) < 2^64 mod N (Lemire: exact uniform);
//     accepted iff  z < (uint64)(min(sigmoid(s_j) / sigma_b, 1) * 2^32).
//   A row with no acceptance in PCV_REJECT_MAX_IT proposals (acceptance rate pathologically low) falls back to a
//   sequential inverse-CDF scan in double precision driven by word w of proposal 0.
#include "pcv_common.cuh"

namespace pcv {

constexpr uint32_t PCV_STREAM_REJECT = 4;
constexpr int PCV_REJECT_MAX_IT = 1024;
constexpr int PCV_REJECT_BATCH = 4;      // proposals evaluated together (independent loads in flight)

template <int D>
__device__ __forceinline__ float chain_score(const float *__restrict__ q, const float *__restrict__ w) {
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < D; k += 4) {
    const float4 v = __ldg(reinterpret_cast<const float4 *>(w + k));
    s = fmaf(q[k], v.x, s);
    s = fmaf(q[k + 1], v.y, s);
    s = fmaf(q[k + 2], v.z, s);
    s = fmaf(q[k + 3], v.w, s);
  }
  return s;
}

template <int D>
__global__ void __launch_bounds__(32)
sigmoid_categorical_kernel(const float *__restrict__ W, int64_t n_rows, const float *__restrict__ max_row_norm,
                           const float *__restrict__ Q,
                           int64_t M, uint64_t seed, uint64_t offset, const uint64_t *__restrict__ offset_dev,
                           int64_t *__restrict__ out_idx, int32_t *__restrict__ out_iters) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= M) return;
  if (offset_dev) offset += *offset_dev;
  float q[D];
#pragma unroll
  for (int k = 0; k < D; k += 4) {
    const float4 v = __ldg(reinterpret_cast<const float4 *>(Q + row * D + k));
    q[k] = v.x; q[k + 1] = v.y; q[k + 2] = v.z; q[k + 3] = v.w;
  }
  float ss = 0.f;
#pragma unroll
  for (int k = 0; k < D; ++k) ss = fmaf(q[k], q[k], ss);
  const float sigma_b = pcv_sigmoidf(sqrtf(ss) * __ldg(max_row_norm) * 1.0001f + 1e-6f);
  const uint64_t r = (uint64_t)row + offset;
  const uint64_t N = (uint64_t)n_rows;
  const uint64_t lemire_t = (0ull - N) % N;     // 2^64 mod N
  int64_t pick = -1;
  int it = 0;
  uint32_t w0 = 0;
  for (; it < PCV_REJECT_MAX_IT && pick < 0; it += PCV_REJECT_BATCH) {
    int64_t j[PCV_REJECT_BATCH];
    uint32_t z[PCV_REJECT_BATCH];
    bool valid[PCV_REJECT_BATCH];
    float s[PCV_REJECT_BATCH];
#pragma unroll
    for (int b = 0; b < PCV_REJECT_BATCH; ++b) {
      const Philox4 p = philox4x32_10((uint32_t)(it + b), (uint32_t)r, (uint32_t)(r >> 32), PCV_STREAM_REJECT,
                                      (uint32_t)seed, (uint32_t)(seed >> 32));
      const uint64_t u = ((uint64_t)p.x << 32) | p.y;
      j[b] = (int64_t)__umul64hi(u, N);
      valid[b] = (u * N) >= lemire_t;
      z[b] = p.z;
      if (it + b == 0) w0 = p.w;
    }
#pragma unroll
    for (int b = 0; b < PCV_REJECT_BATCH; ++b) s[b] = chain_score<D>(q, W + j[b] * D);
#pragma unroll
    for (int b = 0; b < PCV_REJECT_BATCH; ++b) {
      const float ratio = fminf(pcv_sigmoidf(s[b]) / sigma_b, 1.0f);
      const uint64_t thr = (uint64_t)(ratio * 4294967296.0f);
      if (pick < 0 && valid[b] && (uint64_t)z[b] < thr) {
        pick = j[b];
        if (out_iters) out_iters[row] = it + b + 1;
      }
    }
  }
  if (pick < 0) {
    // pathological acceptance rate: sequential inverse CDF in double precision (portable, restated in the oracle)
    double total = 0.0;
    for (int64_t jj = 0; jj < n_rows; ++jj) total += (double)pcv_sigmoidf(chain_score<D>(q, W + jj * D));
    const double target = ((double)w0 + 0.5) * (1.0 / 4294967296.0) * total;
    double acc = 0.0;
    pick = n_rows - 1;
    for (int64_t jj = 0; jj < n_rows; ++jj) {
      acc += (double)pcv_sigmoidf(chain_score<D>(q, W + jj * D));
      if (acc >= target) { pick = jj; break; }
    }
    if (out_iters) out_iters[row] = -1;
  }
  out_idx[row] = pick;
}

}  // namespace pcv

using namespace pcv;

extern "C" int pcv_sigmoid_categorical(const pcv_table *th, const float *Q, int64_t M, uint64_t seed, uint64_t offset,
                                       const uint64_t *offset_dev, int64_t *out_idx, int32_t *out_iters,
                                       pcv_stream_t stream) {
  PCV_CHECK_ARG(th && Q && out_idx, "NULL pointer");
  PCV_CHECK_ARG(M > 0, "M must be > 0");
  const Table *t = reinterpret_cast<const Table *>(th);
  PCV_CHECK_ARG(t->row_offset == 0, "the sampler draws over the whole catalog: pass the full table, not a vocab-parallel shard");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned grid = (unsigned)((M + 31) / 32);   // one warp per CTA: rows finish independently, CTAs spread over the SMs
#define PCV_SAMPLE_CASE(DD)                                                                                          \
  case DD:                                                                                                           \
    sigmoid_categorical_kernel<DD><<<grid, 32, 0, st>>>(t->W, t->n_rows, t->max_row_norm_dev(), Q, M, seed, offset, \
                                                         offset_dev, out_idx, out_iters);                            \
    break;
  switch (t->dim) {
    PCV_SAMPLE_CASE(4)
    PCV_SAMPLE_CASE(8)
    PCV_SAMPLE_CASE(16)
    PCV_SAMPLE_CASE(32)
    PCV_SAMPLE_CASE(64)
    PCV_SAMPLE_CASE(128)
    default:
      set_error("pcv_sigmoid_categorical: dim %d unsupported (use 4, 8, 16, 32, 64 or 128)", t->dim);
      return PCV_ERR_UNSUPPORTED;
  }
#undef PCV_SAMPLE_CASE
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}
