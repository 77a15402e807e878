// pcv_api.cu — handles, error reporting, table construction and in-place refresh.
#include <atomic>
#include <cstdarg>
#include <cstring>
#include <new>

#include "table_images.cuh"

namespace pcv {

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int check_arch() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    set_error("no CUDA device is current (libpcv_b200 has no CPU path)");
    return PCV_ERR_CUDA;
  }
  return pcv_device_ok(dev);
}

// F.normalize(p=2, dim=1, eps=1e-12): x / max(||x||_2, eps)   (cvae.py:31)
// One thread per row; the sum of squares is a sequential-k FMA chain (the
// oracle restates the same order).
__global__ void normalize_rows_kernel(const float *__restrict__ W, int64_t n, int dim,
                                      float *__restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float *w = W + i * dim;
  float ss = 0.f;
  for (int k = 0; k < dim; ++k) ss = fmaf(w[k], w[k], ss);
  float nrm = fmaxf(sqrtf(ss), 1e-12f);
  for (int k = 0; k < dim; ++k) out[i * dim + k] = w[k] / nrm;
}

// One pass over the table: max_j |w_j|_2^2 (row sums of squares as a sequential-k FMA chain, the max as an ordered-uint
// atomicMax: norms are >= 0, so the result does not depend on the order) and every packed image the handle holds,
// written through the layouts of table_images.cuh.  D = 0: any dim, no images (pcv_table_create's norm pass, and the
// dims the tensor-core engines do not serve).  Thread = row, grid-stride: one atomic per CTA.
template <int D>
__global__ void __launch_bounds__(256)
table_refresh_kernel(const float *__restrict__ W, int64_t n_rows, int dim, float4 *__restrict__ packed,
                     uint4 *__restrict__ packed_h, float *__restrict__ packed_t, unsigned int *__restrict__ max_ss) {
  __shared__ float wmax[8];
  float m = 0.f;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n_rows; j += (int64_t)gridDim.x * blockDim.x) {
    float ss = 0.f;
    if constexpr (D == 0) {
      for (int k = 0; k < dim; ++k) ss = fmaf(W[j * dim + k], W[j * dim + k], ss);
    } else {
      const float4 *w = reinterpret_cast<const float4 *>(W + j * D);
      constexpr int G = D / 4 < 8 ? D / 4 : 8;   // 16-byte chunks in flight per thread
#pragma unroll 1
      for (int c0 = 0; c0 < D / 4; c0 += G) {
        float4 v[G];
#pragma unroll
        for (int c = 0; c < G; ++c) v[c] = __ldg(w + c0 + c);
#pragma unroll
        for (int c = 0; c < G; ++c) {
          ss = fmaf(v[c].x, v[c].x, ss); ss = fmaf(v[c].y, v[c].y, ss);
          ss = fmaf(v[c].z, v[c].z, ss); ss = fmaf(v[c].w, v[c].w, ss);
          const int ch = c0 + c;
          packed[sw32_chunk_index(j, ch >> 1, ch & 1, D / 8)] = v[c];
          if (packed_t) {
            packed_t[wt_index<D>(j, 4 * ch + 0)] = v[c].x;
            packed_t[wt_index<D>(j, 4 * ch + 1)] = v[c].y;
            packed_t[wt_index<D>(j, 4 * ch + 2)] = v[c].z;
            packed_t[wt_index<D>(j, 4 * ch + 3)] = v[c].w;
          }
        }
        if constexpr (D == 8)
          if (packed_h) h16_store_row(packed_h, j, v[0], v[1]);
      }
    }
    m = fmaxf(m, ss);
  }
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = fmaxf(m, wmax[w]);
    atomicMax(max_ss, __float_as_uint(m));
  }
}

// max|w| = sqrt(max |w_j|^2) * (1 + 1e-6) into the handle's device scalar; re-arms the running max for the next pass
__global__ void table_norm_finalize_kernel(unsigned int *norm_dev) {
  const float m2 = __uint_as_float(norm_dev[0]);
  reinterpret_cast<float *>(norm_dev)[1] = sqrtf(m2) * 1.000001f;
  norm_dev[0] = 0u;
}

// Both passes on `st`: no allocation, no synchronisation, so a CUDA graph may capture them.
static int table_refresh_launch(Table *t, cudaStream_t st) {
  const int64_t want = (t->n_rows + 255) / 256;
  const int64_t cap = (int64_t)t->sm_count * 8;
  const unsigned grid = (unsigned)(want < cap ? want : cap);
  float4 *p = reinterpret_cast<float4 *>(t->packed);
  uint4 *ph = reinterpret_cast<uint4 *>(t->packed_h);
  switch (t->packed ? t->dim : 0) {
#define PCV_REFRESH_CASE(DD) \
  case DD: table_refresh_kernel<DD><<<grid, 256, 0, st>>>(t->W, t->n_rows, t->dim, p, ph, t->packed_t, t->norm_dev); break;
    PCV_REFRESH_CASE(8)
    PCV_REFRESH_CASE(16)
    PCV_REFRESH_CASE(32)
    PCV_REFRESH_CASE(64)
    PCV_REFRESH_CASE(128)
#undef PCV_REFRESH_CASE
    default: table_refresh_kernel<0><<<grid, 256, 0, st>>>(t->W, t->n_rows, t->dim, nullptr, nullptr, nullptr, t->norm_dev);
  }
  PCV_LAUNCH_CHECK();
  table_norm_finalize_kernel<<<1, 1, 0, st>>>(t->norm_dev);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

__global__ void counter_add_kernel(unsigned long long *c, unsigned long long inc) { *c += inc; }

int table_init_tc(Table *t);  // score_select_tc.cu
void table_free_tc(Table *t);
void table_free_ce(Table *t);   // ce_tc2.cu

}  // namespace pcv

using namespace pcv;

extern "C" {

int pcv_abi_version(void) { return PCV_ABI_VERSION; }
const char *pcv_last_error(void) { return g_err; }
int64_t pcv_launch_count(void) { return g_launches.load(); }

int pcv_counter_add(uint64_t *counter, uint64_t inc, pcv_stream_t stream) {
  PCV_CHECK_ARG(counter != nullptr, "counter is NULL");
  counter_add_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(reinterpret_cast<unsigned long long *>(counter), inc);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

int pcv_device_ok(int device) {
  int major = 0, minor = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device) != cudaSuccess ||
      cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device) != cudaSuccess) {
    cudaGetLastError();
    set_error("pcv_device_ok: cannot query device %d (no CUDA device? this library has no CPU path)", device);
    return PCV_ERR_CUDA;
  }
  if (major != 10) {
    set_error("pcv_device_ok: device %d is sm_%d%d; libpcv_b200 is built for sm_100a only", device, major, minor);
    return PCV_ERR_ARCH;
  }
  return PCV_OK;
}

int pcv_table_create(const float *W, int64_t n_rows, int dim, int64_t row_offset,
                     pcv_table **out) {
  PCV_CHECK_ARG(out != nullptr, "out is NULL");
  *out = nullptr;
  PCV_CHECK_ARG(W != nullptr, "W is NULL");
  PCV_CHECK_ARG(n_rows > 0, "n_rows must be > 0");
  PCV_CHECK_ARG(dim >= 4 && dim <= 128 && dim % 4 == 0, "dim must be a multiple of 4 in [4,128]");
  PCV_CHECK_ARG(((uintptr_t)W & 15) == 0, "W must be 16-byte aligned");
  PCV_CHECK_ARG(row_offset >= 0, "row_offset must be >= 0");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  Table *t = new (std::nothrow) Table();
  PCV_CHECK_ARG(t != nullptr, "out of host memory");
  t->W = W;
  t->n_rows = n_rows;
  t->dim = dim;
  t->row_offset = row_offset;
  t->tmap_valid = 0;
  t->packed = nullptr;
  t->packed_t = nullptr;
  t->packed_h = nullptr;
  t->norm_dev = nullptr;
  cudaGetDevice(&t->device);
  cudaDeviceGetAttribute(&t->sm_count, cudaDevAttrMultiProcessorCount, t->device);
  // one-off: max row norm (error bound of the tf32 filter) into the handle's device scalar, and its host copy (which
  // decides whether the f16 image exists); the refresh re-derives the device scalar with the same two kernels
  {
    cudaError_t e = cudaDeviceSynchronize();  // the table may still be being written on another stream
    if (e == cudaSuccess) e = cudaMalloc(&t->norm_dev, 2 * sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaMemset(t->norm_dev, 0, 2 * sizeof(unsigned int));
    if (e == cudaSuccess) {
      const int64_t want = (n_rows + 255) / 256, cap = (int64_t)t->sm_count * 8;
      table_refresh_kernel<0><<<(unsigned)(want < cap ? want : cap), 256>>>(W, n_rows, dim, nullptr, nullptr, nullptr,
                                                                           t->norm_dev);
      table_norm_finalize_kernel<<<1, 1>>>(t->norm_dev);
      count_launch(2);
      e = cudaMemcpy(&t->max_row_norm, t->max_row_norm_dev(), sizeof(float), cudaMemcpyDeviceToHost);
    }
    if (e != cudaSuccess) {
      cudaGetLastError();
      set_error("pcv_table_create: %s", cudaGetErrorString(e));
      if (t->norm_dev) cudaFree(t->norm_dev);
      delete t;
      return PCV_ERR_CUDA;
    }
  }
  rc = table_init_tc(t);
  if (rc != PCV_OK) {
    table_free_tc(t);
    cudaFree(t->norm_dev);
    delete t;
    return rc;
  }
  *out = reinterpret_cast<pcv_table *>(t);
  return PCV_OK;
}

void pcv_table_destroy(pcv_table *th) {
  Table *t = reinterpret_cast<Table *>(th);
  if (!t) return;
  table_free_tc(t);
  table_free_ce(t);
  if (t->norm_dev) cudaFree(t->norm_dev);
  delete t;
}

int pcv_table_refresh(pcv_table *th, pcv_stream_t stream) {
  PCV_CHECK_ARG(th != nullptr, "t is NULL");
  return table_refresh_launch(reinterpret_cast<Table *>(th), (cudaStream_t)stream);
}

int pcv_normalize_rows(const float *W, int64_t n_rows, int dim, float *out,
                       pcv_stream_t stream) {
  PCV_CHECK_ARG(W && out, "NULL pointer");
  PCV_CHECK_ARG(n_rows > 0 && dim > 0, "bad shape");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  int threads = 256;
  int64_t blocks = (n_rows + threads - 1) / threads;
  normalize_rows_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(W, n_rows, dim, out);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

}  // extern "C"
