// pcv_common.cuh — shared device/host helpers for libpcv_b200.so (sm_100a only).
// Compiled with -fmad=false: every fused multiply-add in this library is an
// explicit fmaf(), so the arithmetic order is the one written and documented
// in DESIGN.md (it is what makes the greedy slates bit-exact, SURVEY F3).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/pcv_b200.h"

namespace pcv {

void set_error(const char *fmt, ...);
void count_launch(int n = 1);
int check_arch();  // PCV_OK when the current device is sm_100-class

struct Table {
  const float *W;
  int64_t n_rows;
  int dim;
  int64_t row_offset;
  int device;
  int sm_count;
  // tcgen05 path: pre-swizzled (SWIZZLE_32B image) copy of W owned by the handle
  float *packed;
  float *packed_t;   // transposed per-tile image for the CE gradient MMA (ce_tc2.cu), built on first use; as large as
                     // the table at D >= 16 (twice at D = 8)
  void *packed_h;    // D = 8: f16 image (8 dims + constant dimension, SWIZZLE_32B) for the f16 filter (score_select_tc.cu)
  int tmap_valid;  // 1 when the tcgen05 engine can serve this table
  float max_row_norm;  // max_j |w_j|_2 (error bound of the tf32 filter) at creation: decides whether packed_h exists
  // device words: [0] running max of |w_j|^2 (ordered uint bits, zero between refreshes), [1] max_j |w_j|_2 as a float,
  // written by pcv_table_create and pcv_table_refresh; the kernels read max|w| from there, never from the host copy
  unsigned int *norm_dev;
  const float *max_row_norm_dev() const { return reinterpret_cast<const float *>(norm_dev + 1); }
  int tc_chunk_tiles;  // tcgen05 filter: tiles per column chunk once the table outgrows the L2
};

#define PCV_CHECK_ARG(cond, msg)                              \
  do {                                                        \
    if (!(cond)) {                                            \
      pcv::set_error("%s: %s", __func__, msg);                \
      return PCV_ERR_ARG;                                     \
    }                                                         \
  } while (0)

#define PCV_CUDA(call)                                                          \
  do {                                                                          \
    cudaError_t _e = (call);                                                    \
    if (_e != cudaSuccess) {                                                    \
      pcv::set_error("%s: %s -> %s", __func__, #call, cudaGetErrorString(_e));  \
      return PCV_ERR_CUDA;                                                      \
    }                                                                           \
  } while (0)

#define PCV_LAUNCH_CHECK()                                                        \
  do {                                                                            \
    cudaError_t _e = cudaGetLastError();                                          \
    if (_e != cudaSuccess) {                                                      \
      pcv::set_error("%s: kernel launch -> %s", __func__, cudaGetErrorString(_e)); \
      return PCV_ERR_CUDA;                                                        \
    }                                                                             \
    pcv::count_launch();                                                          \
  } while (0)

// Packed fp32x2 FMA (Blackwell FFMA2): two independent IEEE fused multiply-adds per instruction on
// 64-bit register pairs, bit-identical to two fmaf().  A {w, w} pair compiles to the instruction's
// scalar-broadcast operand form, so pairing costs no extra instructions.
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float &lo, float &hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ void ffma2(unsigned long long &acc, unsigned long long a, unsigned long long b) {
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b));
}

// ---------------------------------------------------------------------------
// Portable transcendental: the same sequence of IEEE operations is restated in
// oracle/pcv_oracle.c, so exp() agrees bit for bit between the CUDA path and
// the CPU oracle (needed by the reparameterisation and the exponential race).
// Cody-Waite reduction + degree-5 polynomial (Cephes expf coefficients).
// ---------------------------------------------------------------------------
__host__ __device__ __forceinline__ float pcv_expf(float x) {
  x = fminf(fmaxf(x, -86.0f), 88.0f);
  const float magic = 12582912.0f;  // 1.5 * 2^23: adds round-to-nearest-even to integer
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
  union {
    uint32_t u;
    float f;
  } s;
  s.u = (uint32_t)(ni + 127) << 23;
  return e * s.f;
}

// sigmoid(x) = 1 / (1 + exp(-x)), IEEE division (no fast-math in this library).
__host__ __device__ __forceinline__ float pcv_sigmoidf(float x) {
  return 1.0f / (1.0f + pcv_expf(-x));
}

// ---------------------------------------------------------------------------
// Philox4x32-10 counter RNG (Salmon et al., SC'11).  Restated in the oracle and
// pinned there against the Random123 known-answer vectors.
// ---------------------------------------------------------------------------
struct Philox4 {
  uint32_t x, y, z, w;
};

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1,
                                                          uint32_t c2, uint32_t c3,
                                                          uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
  const uint32_t W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)M0 * c0;
    uint64_t p1 = (uint64_t)M1 * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  Philox4 o = {c0, c1, c2, c3};
  return o;
}

// 24-bit uniform in the open interval (0, 1): exact in fp32.
__host__ __device__ __forceinline__ float pcv_u01(uint32_t bits) {
  return ((float)(bits >> 8) + 0.5f) * 5.9604644775390625e-8f;  // 2^-24
}

// Stream ids keep the library's Philox consumers disjoint (counter word 3).  The values are part of every draw:
// changing one changes the eps / mask noise of a given (seed, offset).
enum : uint32_t { PCV_STREAM_NORMAL = 2, PCV_STREAM_BERNOULLI = 3 };

#ifdef __CUDACC__
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Order-preserving int64 key of a (score, global index < 2^32) pair: key = (order-preserving float bits << 32) |
// (0xffffffff - index), top bit flipped, so that the SIGNED 64-bit maximum is the better pair (largest value, equal
// values -> lowest index: torch.max first-index semantics, SURVEY F2).  -0 is packed as +0 so that equal scores compare equal.  No score packs to
// PCV_KEY_NONE (it would be a NaN), which marks an empty list entry.
constexpr long long PCV_KEY_NONE = (long long)0x8000000000000000ull;
__device__ __forceinline__ long long pcv_pack_key(float v, int64_t idx) {
  uint32_t b = __float_as_uint(v + 0.0f);
  b = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  const unsigned long long k = ((unsigned long long)b << 32) | (uint32_t)(0xffffffffu - (uint32_t)idx);
  return (long long)(k ^ 0x8000000000000000ull);
}
__device__ __forceinline__ float pcv_unpack_key(long long key, int64_t &idx) {
  const unsigned long long k = (unsigned long long)key ^ 0x8000000000000000ull;
  uint32_t b = (uint32_t)(k >> 32);
  b = (b & 0x80000000u) ? (b & 0x7fffffffu) : ~b;
  idx = (int64_t)(0xffffffffu - (uint32_t)k);
  return __uint_as_float(b);
}
#endif

}  // namespace pcv
