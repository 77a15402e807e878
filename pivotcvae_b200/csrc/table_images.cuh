// table_images.cuh — where one element of the item table lands in each packed image a table handle owns.
// The packers of pcv_table_create (pack_sw32_kernel, pack_h16_kernel) and of the first tf32 CE call (pack_wt_kernel)
// and the in-place refresh (table_refresh_kernel) all write through these, so the layouts have one definition.
#pragma once
#include <cuda_fp16.h>

#include "tc_common.cuh"

namespace pcv {

// Pre-swizzled tf32 image (score_select_tc.cu): per 256-row tile and k-atom a (8 consecutive fp32 of a row) a
// [256][32 B] block in which the two 16-byte chunks of a row are swapped when bit 2 of the row index is set
// (Swizzle<1,4,3>: address bit 4 ^= bit 7); the ka atoms of a tile follow each other.  -> float4 index of chunk c (0, 1)
// of atom a of row j.
__device__ __forceinline__ int64_t sw32_chunk_index(int64_t j, int a, int c, int ka) {
  return ((j >> 8) * ka + a) * (TC_BN * 2) + (j & (TC_BN - 1)) * 2 + (c ^ (int)((j >> 2) & 1));
}

// f16 image of a D = 8 table (the f16 select filter): row j = 16 f16 (8 dimensions, then the constant dimension 1 and
// zeros) = 32 B, the two 16-byte halves swapped when bit 2 of the row index is set (the same SWIZZLE_32B rule).
// A row holding a NaN is stored as zeros: an f16 NaN pattern would win the filter's unsigned 16-bit chunk maxima and
// hide the real winner of its chunk; as zeros its approximate score is the constant 1, and the refine re-scores it.
__device__ __forceinline__ void h16_store_row(uint4 *__restrict__ out, int64_t j, float4 w0, float4 w1) {
  if (isnan(w0.x + w0.y + w0.z + w0.w + w1.x + w1.y + w1.z + w1.w)) {   // (inf - inf rows: out of the f16 range anyway)
    w0 = make_float4(0.f, 0.f, 0.f, 0.f);
    w1 = w0;
  }
  const __half2 h0 = __floats2half2_rn(w0.x, w0.y), h1 = __floats2half2_rn(w0.z, w0.w);
  const __half2 h2 = __floats2half2_rn(w1.x, w1.y), h3 = __floats2half2_rn(w1.z, w1.w);
  const uint4 lo = make_uint4(*reinterpret_cast<const uint32_t *>(&h0), *reinterpret_cast<const uint32_t *>(&h1),
                              *reinterpret_cast<const uint32_t *>(&h2), *reinterpret_cast<const uint32_t *>(&h3));
  const uint4 hi = make_uint4(0x00003C00u, 0u, 0u, 0u);
  const int sw = (int)((j >> 2) & 1);
  out[2 * j + (0 ^ sw)] = lo;
  out[2 * j + (1 ^ sw)] = hi;
}

// Transposed image of the tf32 CE (ce_tc2.cu, the gradient MMA's B operand): per BN-item tile, BN / 8 k-atoms (8 items
// each) of [NG rows x 32 B]: row r < D = embedding dimension r (rows D..15 zero at D = 8); the two 16-byte chunks of a
// row are swapped when bit 2 of r is set (SWIZZLE_32B).  Padding rows and the tail of the last tile stay zero.
template <int D>
struct WtGeom {
  static constexpr int BN = D <= 32 ? 128 : D == 64 ? 64 : 32;   // items per tile
  static constexpr int NG = D < 16 ? 16 : D;                     // rows of a k-atom (N of the gradient MMA)
};
// -> float index of element (item j, dimension r)
template <int D>
__device__ __forceinline__ int64_t wt_index(int64_t j, int r) {
  using G = WtGeom<D>;
  const int64_t tile = j / G::BN;
  const int i = (int)(j % G::BN), a = i >> 3, c = (i >> 2) & 1, e = i & 3;
  return ((tile * (G::BN / 8) + a) * G::NG + r) * 8 + ((c ^ ((r >> 2) & 1)) << 2) + e;
}

// Error scale of the select filters from the table's max|w| (read from the handle's device scalar): the tf32 filter's
// band is twice 1.25 * 2^-9 * |q| * max|w|; the f16 filter scales query rows by max|w| (+0.3 %).
__device__ __forceinline__ float tc_band_scale(bool f16, float max_row_norm) {
  return f16 ? max_row_norm * 1.003f : 2.0f * 1.25f * 0.001953125f * max_row_norm;
}
// The f16 filter's products fit f16 only while 0 < max|w| < 1e4 (pcv_table_create builds its image only then).  A
// handle refreshed out of that range keeps the image; the filter then hands every stream to the exact re-scan.
__device__ __forceinline__ bool tc_f16_in_range(float max_row_norm) {
  return max_row_norm > 0.f && max_row_norm < 1.0e4f;
}

}  // namespace pcv
