// mlp_tc.cu — fused MLP blocks on the 5th-gen tensor cores (sm_100a), inference engine "tc".
//
// Replaces the same reference code as mlp.cu (pivotcvae.py:159-174, 204-240, 278-291; listcvae.py:106-119;
// cvae.py:79-92; env/response_model.py:76-87): gather / one-hot / concat prologue -> Linear+activation chain ->
// optional reparameterisation, one launch per block (or per chain of two blocks).
//
// The FFMA engines of mlp.cu are bit-identical to the CPU oracle but run at ~10 % of the fp32 peak (latency-bound:
// 8-32 rows per CTA, a cluster barrier per layer).  Here a CTA owns 128 batch rows (= the 128 TMEM lanes) and the
// whole layer chain stays on chip, TMEM-chained:
//
//   layer l accumulates  Y_l[128 x N_l] = X_l[128 x K_l] . W_l^T  in tensor memory (tcgen05.mma kind::tf32, M = 128,
//   N = N_l <= 256, fp32 accumulators; two 256-column regions ping-pong between consecutive layers);
//   8 transform warps (thread = batch row, two groups of four) read Y_l 32 columns at a time (tcgen05.ld), add the
//   bias, apply the activation, split the fp32 result into tf32 hi + lo and write it as a [128 x 32] K-major
//   SWIZZLE_128B chunk into a double-buffered shared-memory operand buffer: that chunk is 32 k-columns of X_{l+1},
//   and layer l+1's MMAs on it start at once while the next chunk is being transformed.  The activations never exist
//   as a whole outside TMEM (a 128 x 256 fp32 tile split in hi/lo would be 256 KB: it does not fit shared memory),
//   nothing goes to HBM between layers;
//   a TMA warp streams the weights, pre-split and pre-swizzled by pcv_mlp_tc_pack into the [N][32] hi | lo images of
//   each 32-k chunk (one bulk copy per chunk, 2 x 64 KB ring).
// (Splitting a row tile's columns over a cluster of CTAs was built and measured first: the all-gather of the operand
// chunks through distributed shared memory moves 3 x 32 KB per chunk at ~20 B/clk/SM — slower than the MMAs it saves.)
//
// Precision: "3xTF32" — lo*hi + hi*lo + hi*hi with hi = rna_tf32(x), lo = rna_tf32(x - hi): products good to ~2^-21.
// The tensor core TRUNCATES its fp32 accumulator on every MMA (measured, profiles/probe_tc_accum.py: a bias of about
// -0.75 x 2^-24 of the accumulator per accumulating MMA; the 96 interleaved MMAs of a 256-deep layer cost -4e-6, 15x
// the error of an fp32 FMA chain).  Layers deeper than 64 therefore run in TWO PASSES over their operand chunks: first
// every small term (lo*hi, hi*lo — while the accumulator is ~2^-11 of its final size their truncations are
// negligible), then the 32 hi*hi MMAs; the transform warps simply produce the chunks twice (the second time hi only).
// Layers at most 64 wide (heads, last layers) have room for FOUR accumulators per output in their TMEM region instead:
// slot 0 takes the small terms, slots 1-3 the hi*hi terms round-robin, the reader adds them in fp32 round-to-nearest
// (one pass, ~1.1x the error of the FMA chain).
// Result: fp32-grade (a few times the distance an fp32 FMA chain has from exact), NOT bit-identical to the oracle's
// sequential chain; the tests hold this engine to the reference fixtures (logits 1e-4, identical slates).
#include "mlp_common.cuh"
#include "tc_common.cuh"

namespace pcv {

constexpr int MT_BM = 128;                  // batch rows per CTA (TMEM lanes)
constexpr int MT_KC = 32;                   // k-chunk: 32 fp32 = one 128-byte swizzle row
constexpr int MT_MAXN = 256;                // widest layer (one TMEM region)
constexpr int MT_MAXK0 = 64;                // widest assembled input (two operand chunks = both operand buffers)
constexpr int MT_MAXCLICKS = 16;            // one-hot segment: clicks per row the prologue handles
// PCV_MLP_AUTO takes this engine from this many batch rows: a CTA owns 128 rows and takes ~30 us per block whatever
// the batch, while the FFMA cluster engine spreads 1024 rows over 128 CTAs in ~18 us but needs ~50 us at 4096 rows
// and ~180 us at 16384.
constexpr int64_t MT_AUTO_MIN_ROWS = 2048;
constexpr int MT_TWOPASS_K = 64;            // layers deeper than this: small terms first, then hi*hi (see above)
constexpr int MT_SLOT_N = 64;               // layers at most this wide keep FOUR accumulators per output in their 256-column
constexpr int MT_NSLOT = 4;                 // region instead (slot 0: small terms, slots 1-3: hi*hi round-robin; added in fp32 RN
                                            // by the reader): one pass, and about the error of an fp32 FMA chain
constexpr int MT_STAGES = 2;                // weight ring
constexpr uint32_t MT_STAGE_BYTES = MT_MAXN * 128 * 2;   // [hi | lo] images of a [256][32] weight chunk
constexpr uint32_t MT_AHALF_BYTES = MT_BM * 128;         // one [128][32] image
constexpr uint32_t MT_ABUF_BYTES = 2 * MT_AHALF_BYTES;   // [hi | lo]
constexpr int MT_NABUF = 2;
constexpr int MT_XWARPS = 8;                // transform warps: two groups of four (one warp per TMEM lane quarter)
constexpr int MT_THREADS = 64 + 32 * MT_XWARPS;
constexpr size_t MT_SMEM = (size_t)MT_STAGES * MT_STAGE_BYTES + (size_t)MT_NABUF * MT_ABUF_BYTES + 1024;

__host__ __device__ __forceinline__ int mt_pad16(int n) { return (n + 15) & ~15; }
__host__ __device__ __forceinline__ int mt_chunks(int kpad) { return (kpad + MT_KC - 1) / MT_KC; }
// accumulation plan of a layer (kpad deep, npad wide)
__host__ __device__ __forceinline__ bool mt_slotted(int npad) { return npad <= MT_SLOT_N; }
__host__ __device__ __forceinline__ int mt_passes(int kpad, int npad) { return (!mt_slotted(npad) && kpad > MT_TWOPASS_K) ? 2 : 1; }
__host__ __device__ __forceinline__ int64_t mt_packed_floats(int n_in, int n_out) {
  return (int64_t)mt_chunks(mt_pad16(n_in)) * mt_pad16(n_out) * 64;
}

__device__ __forceinline__ uint32_t tf32_rna(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return u;
}

// Weight images: chunk c (k = 32c .. 32c+31) = [hi: Npad x 128 B][lo: Npad x 128 B], row n = 32 floats whose
// 16-byte units are XOR-swizzled with (n & 7) (the K-major SWIZZLE_128B layout); rows >= n_out and k >= n_in are zero.
__global__ void mlp_tc_pack_kernel(const float *__restrict__ W, int K, int NO, float *__restrict__ out, int64_t total) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const int npad = mt_pad16(NO);
  const int64_t per_chunk = (int64_t)npad * 64;
  const int c = (int)(e / per_chunk);
  const int rem = (int)(e - (int64_t)c * per_chunk);
  const int half = rem / (npad * 32);
  const int p = rem - half * npad * 32;
  const int n = p >> 5, pos = p & 31;
  const int unit = (pos >> 2) ^ (n & 7);
  const int k = c * MT_KC + unit * 4 + (pos & 3);
  const float v = (n < NO && k < K) ? W[(int64_t)n * K + k] : 0.f;
  const float hi = __uint_as_float(tf32_rna(v));
  out[e] = half ? __uint_as_float(tf32_rna(v - hi)) : hi;
}

#ifdef PCV_TC_TRACE
// CTA 0: role 0 = first transform warp, role 1 = MMA warp; clock64 stamps (profiles/trace_mlp_tc.py)
__device__ long long g_mt_trace[2][64];
#define MT_TRACE(role, i) do { if (blockIdx.x == 0 && lane == 0 && warp == ((role) == 0 ? 2 : 1) && (i) < 64) g_mt_trace[role][i] = clock64(); } while (0)
#else
#define MT_TRACE(role, i) do { } while (0)
#endif

struct MtBars {
  unsigned long long wfull[MT_STAGES], wempty[MT_STAGES], afull[MT_NABUF], aempty[MT_NABUF], accfull;
  uint32_t tmem_base;
};

__device__ __forceinline__ uint64_t mt_desc_sw128(uint32_t saddr) {
  uint64_t d = (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;            // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;  // stride byte offset between 8-row groups
  d |= (uint64_t)1 << 46;            // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;            // LayoutType::SWIZZLE_128B
  return d;
}

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void st_shared_f32(uint32_t addr, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ float ld_shared_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ float4 ld_shared_v4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
// branch-free activation: v > 0 ? v : slope * v (slope 1 / 0.01 / 0 = none / LeakyReLU / ReLU)
__device__ __forceinline__ float mt_act(float v, float slope) { return v > 0.f ? v : v * slope; }

__global__ void __launch_bounds__(MT_THREADS, 1)
mlp_tc_kernel(const __grid_constant__ MlpParams2 P2, int n_blocks, int64_t B) {
  extern __shared__ unsigned char mt_smem_raw[];
  unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(mt_smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t stage0 = smem_u32(smem);
  const uint32_t abuf0 = stage0 + MT_STAGES * MT_STAGE_BYTES;
  __shared__ MtBars Bq;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t b0 = (int64_t)blockIdx.x * MT_BM;
  MT_TRACE(1, 61);

  if (threadIdx.x == 0) {
    for (int s = 0; s < MT_STAGES; ++s) { mbar_init(&Bq.wfull[s], 1); mbar_init(&Bq.wempty[s], 1); }
    // afull: one elected arrive per producing warp (every operand chunk is written by four warps)
    for (int a = 0; a < MT_NABUF; ++a) { mbar_init(&Bq.afull[a], 4); mbar_init(&Bq.aempty[a], 1); }
    mbar_init(&Bq.accfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&Bq.tmem_base)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = Bq.tmem_base;
  MT_TRACE(1, 62);

  if (warp == 0) {
    // ---------------- weight producer ----------------
    // cold start (e.g. after other work evicted them): request the weight images of the whole launch into L2, the
    // CTAs taking turns over the 128-byte lines
    for (int blk = 0; blk < n_blocks; ++blk) {
      const pcv_mlp_desc &d = blk ? P2.b.d : P2.a.d;
      for (int l = 0; l < d.n_layers; ++l) {
        const char *src = reinterpret_cast<const char *>(d.layer[l].Wt);
        const int64_t lines = mt_packed_floats(d.layer[l].n_in, d.layer[l].n_out) / 32;
        for (int64_t i = (int64_t)blockIdx.x * 32 + lane; i < lines; i += (int64_t)gridDim.x * 32)
          asm volatile("prefetch.global.L2 [%0];" ::"l"(src + i * 128));
      }
    }
    if (lane == 0) {
      uint32_t gw = 0;
      for (int blk = 0; blk < n_blocks; ++blk) {
        const pcv_mlp_desc &d = blk ? P2.b.d : P2.a.d;
        for (int l = 0; l < d.n_layers; ++l) {
          const int npad = mt_pad16(d.layer[l].n_out), kpad = mt_pad16(d.layer[l].n_in);
          const int nch = mt_chunks(kpad);
          const int passes = mt_passes(kpad, npad);
          const float *src = d.layer[l].Wt;
          for (int p = 0; p < passes; ++p) {
            const uint32_t bytes = (uint32_t)npad * (p == 0 ? 256u : 128u);   // second pass: the hi image only
            for (int c = 0; c < nch; ++c, ++gw) {
              const uint32_t s = gw % MT_STAGES;
              mbar_wait(&Bq.wempty[s], ((gw / MT_STAGES) & 1) ^ 1);
              mbar_expect_tx(&Bq.wfull[s], bytes);
              tma_bulk_load(smem + (size_t)s * MT_STAGE_BYTES, src + (int64_t)c * npad * 64, bytes, &Bq.wfull[s]);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer (the whole warp, converged; one elected lane issues: tc_common.cuh) ----------------
    uint32_t ga = 0, gw = 0, gl = 0;
    for (int blk = 0; blk < n_blocks; ++blk) {
      const pcv_mlp_desc &d = blk ? P2.b.d : P2.a.d;
      for (int l = 0; l < d.n_layers; ++l, ++gl) {
        const int kpad = mt_pad16(d.layer[l].n_in), npad = mt_pad16(d.layer[l].n_out);
        const int nch = mt_chunks(kpad);
        const int passes = mt_passes(kpad, npad);
        const bool slotted = mt_slotted(npad);
        const uint32_t nmain = (uint32_t)min(MT_NSLOT - 1, kpad >> 3);   // hi*hi slots in use (a 16-deep layer has two k-steps)
        uint32_t written = 0, slot = 1;   // slotted layers: bit s = slot s holds data of this layer
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(npad >> 3) << 17) | ((uint32_t)(MT_BM >> 4) << 24);
        const uint32_t tacc = tmem + (gl & 1) * MT_MAXN;
        uint32_t acc = 0;     // the layer's first MMA overwrites the accumulator
        for (int p = 0; p < passes; ++p) {
          for (int c = 0; c < nch; ++c, ++ga, ++gw) {
            const uint32_t ab = ga & 1, s = gw % MT_STAGES;
            mbar_wait(&Bq.afull[ab], (ga >> 1) & 1);
            if (c == 0 && p == 0) MT_TRACE(1, blk * 26 + 4 + 6 * l);
            if (blk == 0 && l == 1) MT_TRACE(1, 20 + p * 8 + c);            // operand chunk seen (cadence of the deep layer)
            mbar_wait(&Bq.wfull[s], (gw / MT_STAGES) & 1);
            if (blk == 0 && l == 1) MT_TRACE(1, 40 + p * 8 + c);            // weights seen
            if (c == 0 && p == 0) MT_TRACE(1, blk * 26 + 5 + 6 * l);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t a_hi = abuf0 + ab * MT_ABUF_BYTES, w_hi = stage0 + s * MT_STAGE_BYTES;
            // descriptors of the chunk's first k-step; a k-step (8 fp32 = 32 B inside the 128-byte swizzle row) adds 2 to
            // the encoded start address
            uint64_t dah = mt_desc_sw128(a_hi), dal = mt_desc_sw128(a_hi + MT_AHALF_BYTES);
            uint64_t dbh = mt_desc_sw128(w_hi), dbl = mt_desc_sw128(w_hi + (uint32_t)npad * 128u);
            const int atoms = min(4, (kpad - c * MT_KC) >> 3);
#pragma unroll 1
            for (int j = 0; j < atoms; ++j) {
              if (slotted) {
                umma_tf32_elect(tacc, dal, dbh, idesc, written & 1u);
                umma_tf32_elect(tacc, dah, dbl, idesc, 1);
                umma_tf32_elect(tacc + slot * MT_SLOT_N, dah, dbh, idesc, (written >> slot) & 1u);
                written |= 1u | (1u << slot);
                slot = (slot == nmain) ? 1u : slot + 1u;
              } else {
                if (passes == 1 || p == 0) {
                  umma_tf32_elect(tacc, dal, dbh, idesc, acc);
                  umma_tf32_elect(tacc, dah, dbl, idesc, 1);
                  acc = 1;
                }
                if (passes == 1 || p == 1) umma_tf32_elect(tacc, dah, dbh, idesc, 1);
              }
              dah += 2; dal += 2; dbh += 2; dbl += 2;
            }
            umma_commit_elect(&Bq.wempty[s]);
            umma_commit_elect(&Bq.aempty[ab]);
            if (c == 0 && p == 0) MT_TRACE(1, blk * 26 + 6 + 6 * l);
          }
        }
        umma_commit_elect(&Bq.accfull);
        MT_TRACE(1, blk * 26 + 7 + 6 * l);
      }
    }
  } else {
    // ---------------- transform warps: thread = batch row = TMEM lane ----------------
    const int xw = warp - 2;                     // 0..7
    const int grp = xw >> 2;                     // group g produces the operand chunks with (sequence number & 1) == g
    const int quarter = warp & 3;                // TMEM lane quarter = warp id % 4
    const int r = quarter * 32 + lane;
    const int64_t b = b0 + r;
    const uint32_t rowoff = (uint32_t)r * 128u, sw = (uint32_t)r & 7u;
    const uint32_t lane_base = tmem + ((uint32_t)(quarter * 32) << 16);
    uint32_t ga = 0, gl = 0;
    auto acquire = [&](uint32_t g) {   // operand buffer of production g is free: the MMAs of production g - 2 have read it
      mbar_wait(&Bq.aempty[g & 1], ((g >> 1) & 1) ^ 1);
    };
    auto publish = [&](uint32_t g) {   // this warp's rows of production g are in place
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(&Bq.afull[g & 1]);
    };
    for (int blk = 0; blk < n_blocks; ++blk) {
      const MlpParams &P = blk ? P2.b : P2.a;
      const pcv_mlp_desc &d = P.d;
      const int k0pad = mt_pad16(P.n_in0);
      const int nch0 = mt_chunks(k0pad);
      MT_TRACE(0, blk * 26 + 0);
      {
        // ---- prologue: x0 = [segments] for the CTA's 128 rows.
        // Pass 1 (all eight warps): warp w takes rows w, w + 8, ...; lane = element of the 32-wide chunk, so a lane's
        // segment is fixed and its 16 rows' loads are independent: all of them are in flight together (two dependent
        // round trips for a gather: index, then table row) instead of one round trip per element.
        if (blk > 0) {
          // block b reads what block a's epilogue wrote for the same batch rows (z), by other threads of the CTA
          __threadfence_block();
          asm volatile("bar.sync 1, 256;" ::: "memory");
        }
        for (int c = 0; c < nch0; ++c) acquire(ga + c);
        MT_TRACE(0, blk * 26 + 1);
        int oh_seg = -1;                   // the one-hot segment is filled by the row's own thread in pass 2
        for (int s = 0; s < d.n_segments; ++s)
          if (d.seg[s].kind == PCV_SEG_ONEHOT) oh_seg = s;
        // this lane's element of chunk 0 and of chunk 1: segment kind, source pointers (both chunks' loads are issued
        // before either is consumed)
        int kind[2];
        const float *src[2];
        const int64_t *ip[2];
        int64_t rs[2], is[2];              // row strides (floats / indices per batch row)
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          kind[c] = -1; src[c] = nullptr; ip[c] = nullptr; rs[c] = 0; is[c] = 0;
          const int e = c * MT_KC + lane;
          if (c < nch0) {
            for (int s = 0; s < d.n_segments; ++s) {
              if (e >= P.seg_off[s] && e < P.seg_off[s + 1]) {
                const pcv_segment &sg = d.seg[s];
                const int le = e - P.seg_off[s];
                kind[c] = sg.kind;
                if (sg.kind == PCV_SEG_DENSE) {
                  src[c] = (const float *)sg.ptr + le; rs[c] = sg.width;
                } else if (sg.kind == PCV_SEG_GATHER) {
                  const int which = le / sg.width;
                  src[c] = (const float *)sg.ptr + (le - which * sg.width); rs[c] = sg.width;
                  ip[c] = sg.idx + which; is[c] = sg.count;
                }
              }
            }
          }
        }
        if (blk == 0) MT_TRACE(0, 40);
        float v[2][16];
        int64_t gi[2][16];
#pragma unroll
        for (int c = 0; c < 2; ++c)
#pragma unroll
          for (int k = 0; k < 16; ++k) {
            const int64_t bb = b0 + xw + 8 * k;
            v[c][k] = 0.f;
            gi[c][k] = -1;
            if (bb < B) {
              // dense: plain (coherent) loads — it may be what the previous block of this launch wrote
              if (kind[c] == PCV_SEG_DENSE) v[c][k] = __ldcg(src[c] + bb * rs[c]);
              else if (kind[c] == PCV_SEG_GATHER) gi[c][k] = __ldg(ip[c] + bb * is[c]);
            }
          }
#pragma unroll
        for (int c = 0; c < 2; ++c)
#pragma unroll
          for (int k = 0; k < 16; ++k)
            if (gi[c][k] >= 0) v[c][k] = __ldg(src[c] + gi[c][k] * rs[c]);
        if (blk == 0) MT_TRACE(0, 41);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          if (c < nch0) {
            const uint32_t base = abuf0 + ((ga + c) & 1u) * MT_ABUF_BYTES;
#pragma unroll
            for (int k = 0; k < 16; ++k) {
              const uint32_t rr = (uint32_t)(xw + 8 * k);
              st_shared_f32(base + rr * 128u + ((((uint32_t)lane >> 2) ^ (rr & 7u)) << 4) + (((uint32_t)lane & 3u) << 2), v[c][k]);
            }
          }
        }
        // this row's click vector, requested before the barrier so its latency hides behind it
        float rv[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) rv[i] = 0.f;
        if (grp == 0 && oh_seg >= 0 && b < B) {
          const float *rr = (const float *)d.seg[oh_seg].ptr + b * d.seg[oh_seg].count;
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (i < d.seg[oh_seg].count) rv[i] = __ldg(rr + i);
        }
        MT_TRACE(0, blk * 26 + 2);
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (blk == 0) MT_TRACE(0, 42);
        if (grp == 0) {
          // Pass 2 (thread = row): one-hot, normalise, HBM copies, split into tf32 hi | lo
          auto eaddr = [&](int e) {   // raw fp32 staging = the hi image of the chunk
            const uint32_t kk = (uint32_t)e & 31u;
            return abuf0 + ((ga + ((uint32_t)e >> 5)) & 1u) * MT_ABUF_BYTES + rowoff + ((((kk >> 2) ^ sw)) << 4) + ((kk & 3u) << 2);
          };
          if (b < B) {
            if (oh_seg >= 0) {
              float sum = 0.f;
#pragma unroll
              for (int i = 0; i < 16; ++i) sum += rv[i];     // sequential order; + 0 for the padding
              const int hot = (int)sum;  // .to(torch.long) truncates (cvae.py:91)
              if (hot >= 0 && hot <= d.seg[oh_seg].count) st_shared_f32(eaddr(P.seg_off[oh_seg] + hot), 1.f);
            }
            // segment-wide L2 normalisation (F.normalize eps=1e-12), sequential sum order as in mlp.cu
            for (int s = 0; s < d.n_segments; ++s) {
              if (d.seg[s].norm != PCV_NORM_SEGMENT) continue;
              const int off = P.seg_off[s], w = P.seg_off[s + 1] - off;
              float ss = 0.f;
              for (int e = 0; e < w; ++e) { const float x = ld_shared_f32(eaddr(off + e)); ss = fmaf(x, x, ss); }
              const float nrm = fmaxf(sqrtf(ss), 1e-12f);
              for (int e = 0; e < w; ++e) st_shared_f32(eaddr(off + e), ld_shared_f32(eaddr(off + e)) / nrm);
            }
            if (blk == 0) MT_TRACE(0, 43);
            if (d.copy_seg >= 0) {
              const int off = P.seg_off[d.copy_seg], w = P.seg_off[d.copy_seg + 1] - off;
              float *dst = d.out + b * d.out_ld;
              for (int e = 0; e < w; ++e) dst[e] = ld_shared_f32(eaddr(off + e));
            }
          }
          if (blk == 0) MT_TRACE(0, 44);
          for (int c = 0; c < nch0; ++c) {
            const uint32_t base = abuf0 + ((ga + c) & 1u) * MT_ABUF_BYTES + rowoff;
#pragma unroll
            float4 xs[8];
#pragma unroll
            for (uint32_t u = 0; u < 8; ++u) xs[u] = ld_shared_v4(base + ((u ^ sw) << 4));   // bank-conflict-free: rows differ in u ^ sw
#pragma unroll
            for (uint32_t u = 0; u < 8; ++u) {
              const float4 x = xs[u];
              const uint32_t o = (u ^ sw) << 4;
              const uint32_t h0 = tf32_rna(x.x), h1 = tf32_rna(x.y), h2 = tf32_rna(x.z), h3 = tf32_rna(x.w);
              st_shared_v4(base + o, h0, h1, h2, h3);
              st_shared_v4(base + o + MT_AHALF_BYTES, tf32_rna(x.x - __uint_as_float(h0)), tf32_rna(x.y - __uint_as_float(h1)),
                           tf32_rna(x.z - __uint_as_float(h2)), tf32_rna(x.w - __uint_as_float(h3)));
            }
          }
          if (blk == 0) MT_TRACE(0, 45);
          for (int c = 0; c < nch0; ++c) publish(ga + c);
        }
        MT_TRACE(0, blk * 26 + 3);
      }
      ga += nch0;

      for (int l = 0; l < d.n_layers; ++l, ++gl) {
        const pcv_linear &L = d.layer[l];
        const bool last = (l == d.n_layers - 1);
        const int npad = mt_pad16(L.n_out);
        const int nchn = mt_chunks(npad);
        // passes of the NEXT layer, whose operand this layer's output is
        const int passes = last ? 1 : mt_passes(npad, mt_pad16(d.layer[l + 1].n_out));
        const bool slotted = mt_slotted(npad);                           // this layer's accumulators: four slots to add up
        const int nmain = min(MT_NSLOT - 1, mt_pad16(L.n_in) >> 3);
        // 32 accumulator columns from column nb of the layer: (slot1 + slot2 + slot3) + slot0 in fp32 RN, or the single one
        auto read_chunk = [&](uint32_t tbase, int nb, uint32_t (&v)[32]) {
          if (!slotted) {
            TC_LD32(v, tbase + (uint32_t)nb);
            TC_WAIT_LD(v);
          } else {
            uint32_t w[32];
            TC_LD32(v, tbase + (uint32_t)(MT_SLOT_N + nb));
            TC_WAIT_LD(v);
            for (int sidx = 2; sidx <= nmain; ++sidx) {
              TC_LD32(w, tbase + (uint32_t)(sidx * MT_SLOT_N + nb));
              TC_WAIT_LD(w);
#pragma unroll
              for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) + __uint_as_float(w[i]));
            }
            TC_LD32(w, tbase + (uint32_t)nb);
            TC_WAIT_LD(w);
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) + __uint_as_float(w[i]));
          }
        };
        const float slope = L.act == PCV_ACT_LEAKY ? 0.01f : (L.act == PCV_ACT_RELU ? 0.f : 1.f);
        mbar_wait(&Bq.accfull, gl & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t tacc = lane_base + (gl & 1) * MT_MAXN;
        MT_TRACE(0, blk * 26 + 4 + 6 * l);
        if (!last) {
          for (int p = 0; p < passes; ++p) {
            for (int c = 0; c < nchn; ++c) {
              const uint32_t g = ga + (uint32_t)(p * nchn + c);
              if ((int)(g & 1) != grp) continue;
              const int nb = c * MT_KC;
              float bias[32];
#pragma unroll
              for (int i = 0; i < 32; ++i) bias[i] = (nb + i < L.n_out) ? __ldg(L.b + nb + i) : 0.f;
              const bool tr = (blk == 0 && l == 1 && c == 2 && p == 0);
              if (tr) MT_TRACE(0, 50);
              uint32_t v[32];
              read_chunk(tacc, nb, v);
              if (tr) MT_TRACE(0, 51);
              float y[32];
#pragma unroll
              for (int i = 0; i < 32; ++i) y[i] = mt_act(__uint_as_float(v[i]) + bias[i], slope);
              if (tr) MT_TRACE(0, 52);
              acquire(g);
              if (tr) MT_TRACE(0, 53);
              const uint32_t base = abuf0 + (g & 1u) * MT_ABUF_BYTES + rowoff;
#pragma unroll
              for (uint32_t u = 0; u < 8; ++u) {
                const uint32_t h0 = tf32_rna(y[4 * u]), h1 = tf32_rna(y[4 * u + 1]), h2 = tf32_rna(y[4 * u + 2]), h3 = tf32_rna(y[4 * u + 3]);
                const uint32_t o = (u ^ sw) << 4;
                st_shared_v4(base + o, h0, h1, h2, h3);
                if (p == 0)     // the second pass (hi*hi) needs the hi image only
                  st_shared_v4(base + o + MT_AHALF_BYTES, tf32_rna(y[4 * u] - __uint_as_float(h0)), tf32_rna(y[4 * u + 1] - __uint_as_float(h1)),
                               tf32_rna(y[4 * u + 2] - __uint_as_float(h2)), tf32_rna(y[4 * u + 3] - __uint_as_float(h3)));
              }
              if (tr) MT_TRACE(0, 54);
              publish(g);
              if (tr) MT_TRACE(0, 55);
              if (c < 2 && p == 0) MT_TRACE(0, blk * 26 + 5 + 6 * l + c);
            }
          }
          ga += (uint32_t)(passes * nchn);
        } else if (grp == 0) {
          // ---- final epilogue: bias + activation -> out (+ reparameterisation)
          const bool vec = ((d.out_ld | d.out_col0) & 3) == 0 && ((reinterpret_cast<uintptr_t>(d.out) & 15) == 0);
          float *orow = d.out + (b < B ? b : 0) * d.out_ld + d.out_col0;
          for (int nb = 0; nb < L.n_out; nb += 32) {
            float bias[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) bias[i] = (nb + i < L.n_out) ? __ldg(L.b + nb + i) : 0.f;
            uint32_t v[32];
            read_chunk(tacc, nb, v);
            if (b < B) {
#pragma unroll
              for (int i = 0; i < 32; i += 4) {
                float x[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) x[j] = mt_act(__uint_as_float(v[i + j]) + bias[i + j], slope);
                if (vec && nb + i + 4 <= L.n_out) {
                  *reinterpret_cast<float4 *>(orow + nb + i) = make_float4(x[0], x[1], x[2], x[3]);
                } else {
#pragma unroll
                  for (int j = 0; j < 4; ++j)
                    if (nb + i + j < L.n_out) orow[nb + i + j] = x[j];
                }
              }
            }
          }
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          MT_TRACE(0, blk * 26 + 22);
          if (d.latent > 0 && b < B) {
            // cvae.py:79-83: z = eps * exp(0.5 * logvar) + mu; this thread re-reads the [mu | logvar] row it just wrote
            const int Z = d.latent;
            const uint64_t rng_off = d.offset + (d.offset_dev ? *d.offset_dev : 0ull);
            for (int j0 = 0; j0 < Z; j0 += 8) {      // batches of 8 latent columns: all loads first, then the stores
              float mu[8], lv[8], ep[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const bool ok = j0 + i < Z;
                mu[i] = ok ? __ldcg(orow + j0 + i) : 0.f;
                lv[i] = ok ? __ldcg(orow + Z + j0 + i) : 0.f;
                ep[i] = (ok && d.eps) ? __ldg(d.eps + b * Z + j0 + i) : 0.f;
              }
              if (!d.eps) {
#pragma unroll
                for (int i = 0; i < 8; i += 4) {
                  float n4[4];
                  normal4(d.seed, rng_off, b, (j0 + i) >> 2, n4);
                  ep[i] = n4[0]; ep[i + 1] = n4[1]; ep[i + 2] = n4[2]; ep[i + 3] = n4[3];
                }
              }
              float zz[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) zz[i] = ep[i] * pcv_expf(lv[i] * 0.5f) + mu[i];
#pragma unroll
              for (int i = 0; i < 8; ++i)
                if (j0 + i < Z) {
                  d.z[b * Z + j0 + i] = zz[i];
                  if (d.eps_out) d.eps_out[b * Z + j0 + i] = ep[i];
                }
            }
          }
          MT_TRACE(0, blk * 26 + 23);
        }
      }
    }
    MT_TRACE(0, 60);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  MT_TRACE(1, 63);
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem));
  }
}

static bool mlp_tc_fits(const MlpParams *P) {
  const pcv_mlp_desc &d = P->d;
  if (P->n_in0 > MT_MAXK0) return false;
  int n_onehot = 0;
  for (int s = 0; s < d.n_segments; ++s)
    if (d.seg[s].kind == PCV_SEG_ONEHOT) {
      if (++n_onehot > 1 || d.seg[s].count > MT_MAXCLICKS) return false;
    }
  for (int l = 0; l < d.n_layers; ++l)
    if (d.layer[l].n_out > MT_MAXN) return false;
  return true;
}

bool mlp_tc_takes(const MlpParams2 &P, int64_t B, int engine) {
  const bool wanted = engine == PCV_MLP_TC || (engine == PCV_MLP_AUTO && B >= MT_AUTO_MIN_ROWS);
  return wanted && mlp_tc_fits(&P.a) && mlp_tc_fits(&P.b);
}

int mlp_tc_launch(const MlpParams2 &P2, int nblk, int64_t B, cudaStream_t st) {
  int dev = 0;
  cudaGetDevice(&dev);
  static bool attr_set[64] = {false};
  if (!attr_set[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(mlp_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MT_SMEM);
    if (e != cudaSuccess) {
      set_error("pcv_mlp_fwd (tc engine): cudaFuncSetAttribute -> %s", cudaGetErrorString(e));
      return PCV_ERR_CUDA;
    }
    attr_set[dev & 63] = true;
  }
  const int64_t blocks = (B + MT_BM - 1) / MT_BM;
  mlp_tc_kernel<<<(unsigned)blocks, MT_THREADS, MT_SMEM, st>>>(P2, nblk, B);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("pcv_mlp_fwd (tc engine): kernel launch -> %s", cudaGetErrorString(e));
    return PCV_ERR_CUDA;
  }
  count_launch();
  return PCV_OK;
}

}  // namespace pcv

using namespace pcv;

extern "C" {

#ifdef PCV_TC_TRACE
int pcv_debug_mlp_tc_trace(long long *host) {
  return (int)cudaMemcpyFromSymbol(host, g_mt_trace, sizeof(long long) * 2 * 64);
}
#endif

size_t pcv_mlp_tc_packed_bytes(int n_in, int n_out) {
  if (n_in <= 0 || n_out <= 0) return 0;
  return (size_t)mt_packed_floats(n_in, n_out) * sizeof(float);
}

int pcv_mlp_tc_pack(const float *W, int n_in, int n_out, float *packed, pcv_stream_t stream) {
  PCV_CHECK_ARG(W && packed, "NULL pointer");
  PCV_CHECK_ARG(n_in > 0 && n_out > 0 && n_in <= PCV_MAX_WIDTH && n_out <= PCV_MAX_WIDTH, "bad layer shape");
  PCV_CHECK_ARG(((uintptr_t)packed & 127) == 0, "packed buffer must be 128-byte aligned");
  int rc = check_arch();
  if (rc != PCV_OK) return rc;
  const int64_t total = mt_packed_floats(n_in, n_out);
  mlp_tc_pack_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(W, n_in, n_out, packed, total);
  PCV_LAUNCH_CHECK();
  return PCV_OK;
}

}  // extern "C"
