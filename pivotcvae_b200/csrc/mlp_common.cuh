// mlp_common.cuh — descriptors and device helpers shared by the fused MLP engines (mlp.cu: exact FFMA engines,
// mlp_tc.cu: tcgen05 3xTF32 engine).
#pragma once
#include "pcv_common.cuh"

namespace pcv {

constexpr int MLP_KC = 32;    // k-chunk staged per step
constexpr int MLP_NB = 256;   // output columns per pass
constexpr int MLP_WLD_MAX = MLP_NB + 4;   // stage row stride: 257 (CT=1, conflict-free transposing stores) or 260

struct MlpParams {
  pcv_mlp_desc d;
  int n_in0;  // assembled input width
  int ld;     // activation row stride in shared memory (floats)
  int seg_off[PCV_MAX_SEGMENTS + 1];
};

__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == PCV_ACT_LEAKY) return v > 0.f ? v : 0.01f * v;
  if (act == PCV_ACT_RELU) return v > 0.f ? v : 0.f;
  return v;
}

// Philox normals for the reparameterisation (throughput mode): one call gives the
// four eps of latent columns 4c..4c+3 of a row (Box-Muller on two uniform pairs).
__device__ __forceinline__ void normal4(uint64_t seed, uint64_t offset, int64_t row, int c4,
                                        float n[4]) {
  uint64_t r = (uint64_t)row + offset;
  Philox4 p = philox4x32_10((uint32_t)c4, (uint32_t)r, (uint32_t)(r >> 32), PCV_STREAM_NORMAL,
                            (uint32_t)seed, (uint32_t)(seed >> 32));
  float r0 = sqrtf(-2.0f * __logf(pcv_u01(p.x)));
  float r1 = sqrtf(-2.0f * __logf(pcv_u01(p.z)));
  float s0, c0, s1, c1;
  __sincosf(6.283185307179586f * pcv_u01(p.y), &s0, &c0);
  __sincosf(6.283185307179586f * pcv_u01(p.w), &s1, &c1);
  n[0] = r0 * c0; n[1] = r0 * s0; n[2] = r1 * c1; n[3] = r1 * s1;
}

struct MlpParams2 {
  MlpParams a, b;
};

// tensor-core engine (mlp_tc.cu).  mlp_tc_takes: the engine policy (PCV_MLP_*) asks for it at B rows and both blocks
// of P fit it (one block: P.b = P.a); saved outputs are the caller's concern.  nblk = 1 | 2 blocks in the launch.
bool mlp_tc_takes(const MlpParams2 &P, int64_t B, int engine);
int mlp_tc_launch(const MlpParams2 &P2, int nblk, int64_t B, cudaStream_t st);

}  // namespace pcv
