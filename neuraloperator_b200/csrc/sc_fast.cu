// tcgen05 fused transform path (sm_100a).  See DESIGN.md "fast path" for the derivation.
//
// Both transforms are chains of two small GEMMs per 128-row tile, executed on the 5th-generation tensor cores
// with BF16 operands and FP32 accumulation in TMEM.  FP32 accuracy is kept by splitting every operand into
// two bf16 terms (x = x_hi + x_lo, table = T1 + T2) and accumulating the three significant products
// x_hi*T1 + x_lo*T1 + x_hi*T2 ("bf16x3", relative error ~1e-5).
#include <cuda.h>   // CUtensorMap types only; the encoder is fetched with cudaGetDriverEntryPoint (no libcuda link)

#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "sc_fast.h"
#include "sc_half.cuh"
#include "sc_umma.cuh"

namespace sc {

using namespace umma;

// =====================================================================================================
// self-test: D[128 x N] = A[128 x K] * B[N x K]^T with bf16-rounded operands -- exercises the swizzled operand
// stores, the shared-memory / instruction descriptors, TMEM allocation, tcgen05.mma, commit and tcgen05.ld
// exactly the way the transform kernels use them.
// =====================================================================================================
__global__ void __launch_bounds__(128) k_umma_selftest(const float* __restrict__ A, const float* __restrict__ B,
                                                        float* __restrict__ D, int N, int K) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_base;
  uint8_t* sA = smem;
  uint8_t* sB = smem + 128 * K * 2;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (warp == 0) tmem_alloc(&tmem_base, 128);
  if (tid == 0) { mbar_init(&bar, 1); mbar_init_fence(); }
  for (int idx = tid; idx < 128 * K; idx += 128) {
    const int r = idx / K, k = idx % K;
    *reinterpret_cast<__nv_bfloat16*>(sA + sw128_offset(r, k, 128)) = __float2bfloat16_rn(A[idx]);
  }
  for (int idx = tid; idx < N * K; idx += 128) {
    const int r = idx / K, k = idx % K;
    *reinterpret_cast<__nv_bfloat16*>(sB + sw128_offset(r, k, N)) = __float2bfloat16_rn(B[idx]);
  }
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = tmem_base;
  if (tid == 0) {
    const uint32_t idesc = idesc_bf16(128, N);
    for (int ks = 0; ks < K / 16; ++ks) {
      const int slab = ks >> 2, kk = ks & 3;
      const uint64_t da = smem_desc_sw128(smem_u32(sA) + slab * 128 * 128 + kk * 32);
      const uint64_t db = smem_desc_sw128(smem_u32(sB) + slab * N * 128 + kk * 32);
      mma_bf16_ss(tmem, da, db, idesc, ks > 0);
    }
    mma_commit(&bar);
  }
  mbar_wait(&bar, 0);
  tc_fence_after_sync();
  for (int c = 0; c < N; c += 16) {
    float v[16];
    tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + c, v);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 16; ++i) D[(size_t)(warp * 32 + lane) * N + c + i] = v[i];
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 128);
}

// same product with the A operand resident in TENSOR MEMORY (tcgen05.st, then tcgen05.mma with a TMEM A operand)
__global__ void __launch_bounds__(128) k_umma_selftest_ts(const float* __restrict__ A, const float* __restrict__ B,
                                                           float* __restrict__ D, int N, int K) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_base;
  uint8_t* sB = smem;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (warp == 0) tmem_alloc(&tmem_base, 256);
  if (tid == 0) { mbar_init(&bar, 1); mbar_init_fence(); }
  for (int idx = tid; idx < N * K; idx += 128) {
    const int r = idx / K, k = idx % K;
    *reinterpret_cast<__nv_bfloat16*>(sB + sw128_offset(r, k, N)) = __float2bfloat16_rn(B[idx]);
  }
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = tmem_base;
  const uint32_t tm_a = tmem + 128;                          // A: columns 128 .. 128 + K/2
  {
    const int row = warp * 32 + lane;
    for (int c = 0; c < K / 2; c += 16) {
      uint32_t w[16];
#pragma unroll
      for (int e = 0; e < 16; ++e) w[e] = pack_bf16(A[(size_t)row * K + 2 * (c + e)], A[(size_t)row * K + 2 * (c + e) + 1]);
      tmem_st16(tm_a + ((uint32_t)(warp * 32) << 16) + c, w);
    }
    tmem_st_wait();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  if (tid == 0) {
    const uint32_t idesc = idesc_bf16(128, N);
    for (int ks = 0; ks < K / 16; ++ks) {
      const int slab = ks >> 2, kk = ks & 3;
      mma_bf16_ts(tmem, tm_a + ks * 8, smem_desc_sw128(smem_u32(sB) + slab * N * 128 + kk * 32), idesc, ks > 0);
    }
    mma_commit(&bar);
  }
  mbar_wait(&bar, 0);
  tc_fence_after_sync();
  for (int c = 0; c < N; c += 16) {
    float v[16];
    tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + c, v);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 16; ++i) D[(size_t)(warp * 32 + lane) * N + c + i] = v[i];
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 256);
}

bool umma_selftest_ts(const float* A, const float* B, float* D, int N, int K, cudaStream_t st) {
  if (N < 16 || N > 128 || N % 16 != 0 || K < 64 || K > 256 || K % 64 != 0) {
    set_error("umma selftest: need N in 16..128 step 16 and K in 64..256 step 64");
    return false;
  }
  const size_t smem = (size_t)N * K * 2 + 1024;
  if (!cuda_ok(cudaFuncSetAttribute(k_umma_selftest_ts, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
               "cudaFuncSetAttribute(selftest_ts)"))
    return false;
  k_umma_selftest_ts<<<1, 128, smem, st>>>(A, B, D, N, K);
  count_launch();
  return cuda_ok(cudaGetLastError(), "k_umma_selftest_ts launch");
}

bool umma_selftest(const float* A, const float* B, float* D, int N, int K, cudaStream_t st) {
  if (N < 16 || N > 128 || N % 16 != 0 || K < 64 || K > 256 || K % 64 != 0) {
    set_error("umma selftest: need N in 16..128 step 16 and K in 64..256 step 64");
    return false;
  }
  const size_t smem = (size_t)(128 + N) * K * 2 + 1024;
  if (!cuda_ok(cudaFuncSetAttribute(k_umma_selftest, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
               "cudaFuncSetAttribute(selftest)"))
    return false;
  k_umma_selftest<<<1, 128, smem, st>>>(A, B, D, N, K);
  count_launch();
  return cuda_ok(cudaGetLastError(), "k_umma_selftest launch");
}

// =====================================================================================================
// fused analysis:  tile of 128 image rows  ->  kept modes of the G = 128/H images the tile holds
//
//   stage 1 (last dim)    D1[h, j]   = sum_w x[h, w] * TA[w, j]                 M=128 (rows)  N=2*N1  K=W
//   stage 2 (leading dim) D2[i', n]  = sum_{h,p} A2[i', (h,p)] * R_p[h, n]      M=128         N=N1    K=256
//
//   Every role is its own pipeline stage with double buffers in between:
//   warp  18    TMA producer: x slabs [128 rows x 64 fp32] -> two-deep fp32 staging ring (one tensor load per slab)
//   warps 10-17 converters: staging -> bf16 hi/lo split -> swizzled STS into the operand slab
//   warp  8     stage-1 MMA issuer (+ TMEM allocation)          ring slab -> D1[2]
//   warps 4-7   epilogue 1: D1 -> R -> bf16 hi/lo B operand of stage 2 (B2, single buffer)
//   warp  9     stage-2 MMA issuer                                B2 -> D2[2]
//   warps 0-3   epilogue 2: D2 -> kept modes in global memory
// =====================================================================================================
// debug timeline: role r, tile i, phase ph (0 = iteration start, 1 = inputs ready, 2 = work done) of CTA 0
#define SC_TRACE(P, role, i, ph)                                                                        \
  do {                                                                                                  \
    if ((P).trace != nullptr && blockIdx.x == 0 && (threadIdx.x & 31) == 0 && (i) < 16)                \
      (P).trace[(((role) * 16 + (i)) * 4 + (ph))] = clock64();                                          \
  } while (0)

__device__ __forceinline__ void st_global_v8(float* p, const float* v) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
               "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
               : "memory");
}

constexpr int FA_F32_STAGES = 3;   // depth of the fp32 TMA staging ring (32 KB slabs): covers the HBM latency under load
constexpr int FA_LOADER_WARPS = 8;
constexpr int FA_LOADER_ITERS = 128 / (FA_LOADER_WARPS * 2);   // row passes per slab: a loader warp covers 2 rows x 64 floats
constexpr int FA_LOADER_WARP0 = 10;
constexpr int FA_TMA_WARP = FA_LOADER_WARP0 + FA_LOADER_WARPS;          // one extra warp streams x with TMA loads
constexpr int FA_THREADS = (FA_TMA_WARP + 1) * 32;                     // 608
constexpr int FA_SLAB_BYTES = 128 * 128;                                // one [128 x 64] bf16 slab
constexpr int FA_STAGE_BYTES = 2 * FA_SLAB_BYTES;                       // hi + lo

struct AnaParams {
  const float* x;
  float2* out;
  const uint8_t* b1_img;   // [2*N1 x W] bf16, canonical K-major SW128 image (T1 rows then T2 rows)
  const uint8_t* a2_img;   // [128 x 256] bf16, plain row-major: real-embedded leading-dim table (T1 rows 0-63, T2 rows 64-127);
                           // copied once into TENSOR MEMORY and used as the TMEM A operand of every stage-2 MMA
  int n_tiles, W, slabs, N1, KX, QROWS, n_stages, tmem_cols;
  int l2_stream_hint;      // 1: the x slabs are loaded with an L2 evict-first policy (read once)
  int quad_major;          // 1: modes are written in the quad-major layout out[quad][image][4 modes] (contraction operands become
                           //    contiguous 32-byte sectors along the image index), 0: out[image][modes]
  int G, Mt;               // images per tile, kept modes per image
  int qm_tma;              // 1: quad-major output through one tensor store per tile (k_fused_analysis2, one image per tile)
  long long n_images;      // all images of the launch (the quad stride of the quad-major layout, in sectors)
  // Operands of the NEXT kernels of the chain (weights, saved modes) that this launch pulls into L2 while it streams the images:
  // the transform is bound by shared memory, not by DRAM, so the extra reads are free here, whereas the contraction kernels
  // would otherwise wait for them at DRAM latency with 32-byte requests (measured: ~9000 of their ~24000 cycles).
  const uint8_t* pf_ptr[2];
  unsigned long long pf_bytes[2];
  uint32_t off_f32, off_ring, off_b1, off_a2, off_b2, off_scratch, stage_off;   // stage_off: output staging, relative to off_scratch
  long long* trace;        // debug timeline of CTA 0 (SC_TRACE_FILE), else nullptr
};

template <int N1>
__global__ void __launch_bounds__(FA_THREADS, 1) k_fused_analysis(const AnaParams P, const __grid_constant__ CUtensorMap x_map) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // swizzle atoms need 1024-byte alignment
  __shared__ uint64_t bar_full[4], bar_empty[4], bar_d1_full[2], bar_d1_empty[2], bar_b2_full, bar_b2_empty,
      bar_d2_full[2], bar_d2_empty[2], bar_f32_full[FA_F32_STAGES], bar_f32_empty[FA_F32_STAGES];
  __shared__ uint32_t tmem_base_slot;
  constexpr int half = N1 / 2;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int NS = P.n_stages;
  uint8_t* s_b1 = smem + P.off_b1;
  uint8_t* s_b2 = smem + P.off_b2;
  float* s_scr = reinterpret_cast<float*>(smem + P.off_scratch);

  if (tid == 0) {
    for (int i = 0; i < NS; ++i) { mbar_init(&bar_full[i], FA_LOADER_WARPS); mbar_init(&bar_empty[i], 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bar_d1_full[i], 1); mbar_init(&bar_d1_empty[i], 128);
      mbar_init(&bar_d2_full[i], 1); mbar_init(&bar_d2_empty[i], 128);
    }
    for (int i = 0; i < FA_F32_STAGES; ++i) { mbar_init(&bar_f32_full[i], 1); mbar_init(&bar_f32_empty[i], FA_LOADER_WARPS); }
    mbar_init(&bar_b2_full, 128);
    mbar_init(&bar_b2_empty, 1);
    mbar_init_fence();
  }
  if (warp == 8) tmem_alloc(&tmem_base_slot, (uint32_t)P.tmem_cols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  if (warp < FA_LOADER_WARP0) {
    // constant operand images are staged by the consumer-side warps only; the loaders start streaming x at once
    constexpr int NT = FA_LOADER_WARP0 * 32;
    copy_image(s_b1, P.b1_img, (2 * N1 * P.W * 2) / 16, tid, NT);
    if (warp < 4) {   // leading-dim table -> tensor memory: lane = table row, two bf16 K-elements per 32-bit column
      const uint32_t* src = reinterpret_cast<const uint32_t*>(P.a2_img) + (size_t)(warp * 32 + lane) * 128;
      const uint32_t tm_a2_w = tmem_base_slot + (uint32_t)(6 * N1) + ((uint32_t)(warp * 32) << 16);
#pragma unroll 2
      for (int c = 0; c < 128; c += 16) {
        uint32_t w[16];
#pragma unroll
        for (int e = 0; e < 16; e += 4) {
          const uint4 v = __ldg(reinterpret_cast<const uint4*>(src + c + e));
          w[e] = v.x; w[e + 1] = v.y; w[e + 2] = v.z; w[e + 3] = v.w;
        }
        tmem_st16(tm_a2_w + c, w);
      }
      tmem_st_wait();
      tc_fence_before_sync();
    }
    uint4* z = reinterpret_cast<uint4*>(s_b2);   // padding rows of B2 (kx >= KX) stay zero for the whole kernel
    for (int i = tid; i < (N1 * 512) / 16; i += NT) z[i] = make_uint4(0, 0, 0, 0);
    fence_proxy_async_smem();
    asm volatile("bar.sync 2, %0;" ::"n"(NT) : "memory");
  }
  const uint32_t tmem = tmem_base_slot;
  const uint32_t tm_d1[2] = {tmem, tmem + (uint32_t)(2 * N1)};
  const uint32_t tm_d2[2] = {tmem + (uint32_t)(4 * N1), tmem + (uint32_t)(5 * N1)};
  const uint32_t tm_a2 = tmem + (uint32_t)(6 * N1);

  const int n_local = (P.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == FA_TMA_WARP) {
    // ------------------------------------------------------------------ TMA producer: one tensor load per 32 KB slab
    const int total = n_local * P.slabs;
    uint8_t* f32_stage = smem + P.off_f32;
    const uint64_t pol = l2_policy_evict_first();
    pdl_wait();                                  // x is produced by the previous kernel of the stream
    // Hand-over to the next kernel of the stream only AFTER this CTA has seen its own predecessor complete: a kernel of this
    // library may then read, ahead of its own wait, anything its immediate predecessor does not write (the contraction
    // fetches the weights that way).  The dependents still start as soon as this CTA leaves its SM.
    pdl_launch_dependents();
    constexpr unsigned long long PF_PIECE = 8192;
    for (int idx = 0; idx < total; ++idx) {
      const int sb = idx % FA_F32_STAGES;
      mbar_wait(&bar_f32_empty[sb], (uint32_t)(((idx / FA_F32_STAGES) & 1) ^ 1));
      if (elect_one()) {
#pragma unroll
        for (int r = 0; r < 2; ++r) {        // this CTA's idx-th 8 KB piece of each prefetch range
          const unsigned long long off = ((unsigned long long)idx * gridDim.x + blockIdx.x) * PF_PIECE;
          if (off < P.pf_bytes[r]) {
            const unsigned long long left = P.pf_bytes[r] - off;
            bulk_prefetch_l2(P.pf_ptr[r] + off, (uint32_t)(left < PF_PIECE ? left : PF_PIECE));
          }
        }
        const int tile = (int)blockIdx.x + (idx / P.slabs) * (int)gridDim.x, slab = idx % P.slabs;
        mbar_arrive_expect_tx(&bar_f32_full[sb], 32768u);
        if (P.l2_stream_hint) tma_load_2d_hint(f32_stage + sb * 32768, &x_map, &bar_f32_full[sb], slab * 64, tile * 128, pol);
        else
          tma_load_2d(f32_stage + sb * 32768, &x_map, &bar_f32_full[sb], slab * 64, tile * 128);
      }
      __syncwarp();
    }
  } else if (warp >= FA_LOADER_WARP0) {
    // ------------------------------------------------------------------ converters
    // x arrives in a FA_F32_STAGES-deep fp32 staging ring ([128 x 64] fp32 per slab, written by the TMA engine: 64 KB in flight per
    // SM, no registers, no LSU issue slots); each thread splits its 16-byte pieces into bf16 hi/lo operand tiles.
    const int lt = tid - FA_LOADER_WARP0 * 32;
    constexpr int RP = FA_LOADER_WARPS * 2;      // rows covered per pass
    const int rbase = lt >> 4, c4 = lt & 15;     // 16 float4 per 64-float row segment
    uint8_t* f32_stage = smem + P.off_f32;       // two [128 x 64] fp32 slabs, row pitch 256 B
    const uint32_t my_f32 = (uint32_t)(rbase * 256 + c4 * 16);
    uint32_t g = 0;                              // running slab counter
    const int total = n_local * P.slabs;
    for (int idx = 0; idx < total; ++idx, ++g) {
      const int slot = (int)(g % (uint32_t)NS);
      const uint32_t ph = (g / (uint32_t)NS) & 1u;
      const int sb = idx % FA_F32_STAGES;
      if (warp == FA_LOADER_WARP0) SC_TRACE(P, 0, idx, 0);
      mbar_wait(&bar_f32_full[sb], (uint32_t)((idx / FA_F32_STAGES) & 1));
      if (warp == FA_LOADER_WARP0) SC_TRACE(P, 7, idx, 0);
      uint2 hi[FA_LOADER_ITERS], lo[FA_LOADER_ITERS];
      const uint8_t* fsrc = f32_stage + sb * 32768 + my_f32;
#pragma unroll
      for (int it = 0; it < FA_LOADER_ITERS; ++it) {
        const float4 v = *reinterpret_cast<const float4*>(fsrc + it * RP * 256);
        split2_bf16(v.x, v.y, hi[it].x, lo[it].x);
        split2_bf16(v.z, v.w, hi[it].y, lo[it].y);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_f32_empty[sb]);   // this warp has consumed its pieces of the staging buffer
      if (warp == FA_LOADER_WARP0) SC_TRACE(P, 0, idx, 1);
      mbar_wait(&bar_empty[slot], ph ^ 1u);
      if (warp == FA_LOADER_WARP0) SC_TRACE(P, 0, idx, 2);
      uint8_t* shi = smem + P.off_ring + (size_t)slot * FA_STAGE_BYTES;
      uint8_t* slo = shi + FA_SLAB_BYTES;
#pragma unroll
      for (int it = 0; it < FA_LOADER_ITERS; ++it) {
        const uint32_t off = sw128_offset(rbase + it * RP, c4 * 4, 128);
        *reinterpret_cast<uint2*>(shi + off) = hi[it];
        *reinterpret_cast<uint2*>(slo + off) = lo[it];
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_full[slot]);
    }
  } else if (warp == 8) {
    // ------------------------------------------------------------------ stage-1 MMA issuer (warp-uniform, one elected lane issues)
    {
      const uint32_t idesc_p1 = idesc_bf16(128, 2 * N1), idesc_p2 = idesc_bf16(128, N1);
      const uint32_t b1_lo = desc_lo(smem_u32(s_b1)), ring_lo = desc_lo(smem_u32(smem + P.off_ring));
      uint32_t g = 0;
      for (int i = 0; i < n_local; ++i) {
        const int buf = i & 1;
        SC_TRACE(P, 1, i, 0);
        mbar_wait(&bar_d1_empty[buf], (uint32_t)(((i >> 1) & 1) ^ 1));
        tc_fence_after_sync();
        SC_TRACE(P, 1, i, 1);
        for (int s = 0; s < P.slabs; ++s, ++g) {
          const int slot = (int)(g % (uint32_t)NS);
          mbar_wait(&bar_full[slot], (g / (uint32_t)NS) & 1u);
          tc_fence_after_sync();
          const uint32_t d_hi = ring_lo + (uint32_t)slot * (FA_STAGE_BYTES >> 4), d_lo = d_hi + (FA_SLAB_BYTES >> 4);
          const uint32_t d_b = b1_lo + (uint32_t)s * ((2 * N1 * 128) >> 4);
          if (elect_one()) {
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              mma_bf16_ss(tm_d1[buf], desc_from_lo(d_hi + 2 * kk), desc_from_lo(d_b + 2 * kk), idesc_p1, (s | kk) != 0);
              mma_bf16_ss(tm_d1[buf], desc_from_lo(d_lo + 2 * kk), desc_from_lo(d_b + 2 * kk), idesc_p2, true);
            }
            mma_commit(&bar_empty[slot]);
          }
          __syncwarp();
        }
        if (elect_one()) mma_commit(&bar_d1_full[buf]);
        __syncwarp();
        SC_TRACE(P, 1, i, 2);
      }
    }
    __syncwarp();
  } else if (warp == 9) {
    // ------------------------------------------------------------------ stage-2 MMA issuer
    {
      const uint32_t idesc_p2 = idesc_bf16(128, N1);
      const uint32_t b2_lo = desc_lo(smem_u32(s_b2));
      for (int i = 0; i < n_local; ++i) {
        const int buf = i & 1;
        SC_TRACE(P, 3, i, 0);
        mbar_wait(&bar_b2_full, (uint32_t)(i & 1));
        mbar_wait(&bar_d2_empty[buf], (uint32_t)(((i >> 1) & 1) ^ 1));
        tc_fence_after_sync();
        SC_TRACE(P, 3, i, 1);
        if (elect_one()) {
#pragma unroll
          for (int ks = 0; ks < 16; ++ks) {
            const int slab = ks >> 2, kk = ks & 3;
            mma_bf16_ts(tm_d2[buf], tm_a2 + ks * 8, desc_from_lo(b2_lo + slab * ((N1 * 128) >> 4) + 2 * kk), idesc_p2, ks > 0);
          }
          mma_commit(&bar_b2_empty);
          mma_commit(&bar_d2_full[buf]);
        }
        __syncwarp();
        SC_TRACE(P, 3, i, 2);
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ epilogue 1: D1 -> B operand of stage 2
    const int q4 = warp - 4;                                  // TMEM lane quarter; tile row h = q4*32 + lane
    const uint32_t lane_sel = (uint32_t)(q4 * 32) << 16;
    const int KX = P.KX;
    // B2[n][k2], k2 = 2*h + part: row h owns 4 bytes of every row n, inside K-slab q4 (64 columns = 32 rows h)
    uint8_t* b2_mine = s_b2 + q4 * (N1 * 128) + (lane & 3) * 4;
    const int chunk = lane >> 2;
    for (int i = 0; i < n_local; ++i) {
      const int buf = i & 1;
      if (warp == 4) SC_TRACE(P, 2, i, 0);
      mbar_wait(&bar_d1_full[buf], (uint32_t)((i >> 1) & 1));
      mbar_wait(&bar_b2_empty, (uint32_t)((i & 1) ^ 1));
      tc_fence_after_sync();
      if (warp == 4) SC_TRACE(P, 2, i, 1);
#pragma unroll
      for (int c = 0; c < N1; c += 16) {
        float t1[16], t2[16];
        tmem_ld16(tm_d1[buf] + lane_sel + c, t1);        // x_hi*T1 + x_lo*T1
        tmem_ld16(tm_d1[buf] + lane_sel + N1 + c, t2);   // x_hi*T2
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int kx = c / 2 + e;                       // compile-time; slots kx >= KX hold exact zeros (zero table rows)
          uint32_t hi, lo;
          split2_bf16(t1[2 * e] + t2[2 * e], t1[2 * e + 1] + t2[2 * e + 1], hi, lo);
          *reinterpret_cast<uint32_t*>(b2_mine + kx * 128 + ((chunk ^ (kx & 7)) << 4)) = hi;
          *reinterpret_cast<uint32_t*>(b2_mine + (half + kx) * 128 + ((chunk ^ ((half + kx) & 7)) << 4)) = lo;
        }
      }
      tc_fence_before_sync();
      mbar_arrive(&bar_d1_empty[buf]);
      fence_proxy_async_smem();
      mbar_arrive(&bar_b2_full);
      if (warp == 4) SC_TRACE(P, 2, i, 2);
    }
  } else {
    // ------------------------------------------------------------------ epilogue 2: D2 -> kept modes
    const int row = warp * 32 + lane;                        // output row i' (0-63: T1 rows, 64-127: T2 rows)
    const uint32_t lane_sel = (uint32_t)(warp * 32) << 16;
    const int KX = P.KX;
    pdl_wait();                                              // the mode buffer may still be read by the previous kernel
    for (int i = 0; i < n_local; ++i) {
      const int buf = i & 1;
      if (warp == 0) SC_TRACE(P, 4, i, 0);
      mbar_wait(&bar_d2_full[buf], (uint32_t)((i >> 1) & 1));
      tc_fence_after_sync();
      if (warp == 0) SC_TRACE(P, 4, i, 1);
      float d[N1];
#pragma unroll
      for (int c = 0; c < N1; c += 16) tmem_ld16(tm_d2[buf] + lane_sel + c, *reinterpret_cast<float(*)[16]>(&d[c]));
      tmem_ld_wait();
      if (warp == 0) SC_TRACE(P, 5, i, 0);
      tc_fence_before_sync();
      mbar_arrive(&bar_d2_empty[buf]);
      if (warp == 0) SC_TRACE(P, 5, i, 1);
      // T2 rows (warps 2,3) hand hi+lo sums to the matching T1 rows (warps 0,1).  Straight-line code over all N1/2 column
      // slots (padding slots carry exact zeros): runtime bounds checks here turn into a serial LDS->FADD->SHFL->STS chain.
      constexpr int SP = half + 1;                 // scratch row pitch in floats
      if (warp >= 2) {
        float* dst = s_scr + (row - 64) * SP;
#pragma unroll
        for (int kx = 0; kx < half; ++kx) dst[kx] = d[kx] + d[half + kx];
      }
      if (tid == 0) bulk_wait_read_1();            // the block stored two tiles ago has left its staging buffer
      if (warp == 0) SC_TRACE(P, 5, i, 2);
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (warp == 0) SC_TRACE(P, 6, i, 0);
      // the tile's modes are ONE contiguous block of QROWS*KX complex numbers: stage it, then a single bulk async store
      float2* stage = reinterpret_cast<float2*>(smem + P.off_scratch + P.stage_off) + (i & 1) * (P.QROWS * KX);
      if (warp < 2) {
        const float* src = s_scr + row * SP;
        const int q = row >> 1, part = row & 1;
        const bool live = q < P.QROWS && part == 0;
        float mine[half], other[half];
#pragma unroll
        for (int kx = 0; kx < half; ++kx) mine[kx] = d[kx] + d[half + kx] + src[kx];
#pragma unroll
        for (int kx = 0; kx < half; ++kx) other[kx] = __shfl_xor_sync(0xffffffffu, mine[kx], 1);
        float2* my = stage + q * KX;
#pragma unroll
        for (int kx = 0; kx < half; ++kx)
          if (live && kx < KX) my[kx] = make_float2(mine[kx], other[kx]);
      }
      if (warp == 0) SC_TRACE(P, 6, i, 1);
      fence_proxy_async_smem();
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (warp == 0) SC_TRACE(P, 6, i, 2);
      if (P.quad_major) {
        // one 32-byte sector per (image of the tile, quad of modes): element (image, m) lives at ((m >> 2) * n_images + image) * 4 + (m & 3)
        const int tile = (int)blockIdx.x + i * (int)gridDim.x;
        const int nq = P.Mt >> 2;
        for (int idx = tid; idx < P.G * nq; idx += 128) {
          const int g = idx / nq, q = idx - g * nq;
          const float4* sp = reinterpret_cast<const float4*>(stage + g * P.Mt + 4 * q);
          const float4 lo4 = sp[0], hi4 = sp[1];
          const float o8[8] = {lo4.x, lo4.y, lo4.z, lo4.w, hi4.x, hi4.y, hi4.z, hi4.w};
          st_global_v8(reinterpret_cast<float*>(P.out + ((long long)q * P.n_images + (long long)tile * P.G + g) * 4), o8);
        }
      } else if (tid == 0) {
        const int tile = (int)blockIdx.x + i * (int)gridDim.x;
        bulk_store(P.out + (size_t)tile * P.QROWS * KX, stage, (uint32_t)(P.QROWS * KX * 8));
        bulk_commit();
      }
      if (warp == 0) SC_TRACE(P, 4, i, 2);
    }
    if (tid == 0) bulk_wait_all();
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 8) tmem_dealloc(tmem, (uint32_t)P.tmem_cols);
}

// =====================================================================================================
// fused analysis, second generation: the image rows (A operand of stage 1) live in TENSOR MEMORY
//
//   k_fused_analysis is bound by shared-memory bandwidth (per 128-row tile: 64 KB TMA write, 64 KB converter reads, 64 KB of
//   swizzled bf16 hi / lo stores, ~100 KB of stage-1 operand fetches, ...).  Here the converters own image rows (thread <-> TMEM
//   lane), read them from 128-byte-swizzled TMA boxes and write the bf16 hi / lo pairs with tcgen05.st into a two-stage ring of
//   [128 lanes x (32 + 32) columns]; the stage-1 MMAs take A from tensor memory.  That removes the bf16 stores and the A half of
//   the operand fetches (~128 KB of the ~360 KB per tile) and frees the shared memory of the operand ring for a deeper fp32 TMA
//   ring.  Tensor memory: D1[2] 4*N1 | D2 N1 (single-buffered) | leading-dim table 128 | x ring 128  ->  N1 <= 48.
//   Everything downstream of stage 1 is k_fused_analysis unchanged.
// =====================================================================================================
constexpr int FA2_X_STAGES = 2, FA2_MAX_F32 = 6;

// S: storage of x -- 0 float ([128 x 32 floats] boxes, two per slab), SC_FLAG_GRID_F16 / SC_FLAG_GRID_BF16 (one [128 x 64 elements]
// box per slab: the same 128-byte rows and swizzle, half the bytes; the converters widen each element before the hi / lo split,
// so the operands are bit for bit those of the float path on the widened input)
template <int N1, int S>
__global__ void __launch_bounds__(FA_THREADS, 1) k_fused_analysis2(const AnaParams P, const __grid_constant__ CUtensorMap x_map,
                                                                     const __grid_constant__ CUtensorMap qm_map) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // swizzle atoms need 1024-byte alignment
  __shared__ uint64_t bar_full[FA2_X_STAGES], bar_empty[FA2_X_STAGES], bar_d1_full[2], bar_d1_empty[2], bar_b2_full, bar_b2_empty,
      bar_d2_full[1], bar_d2_empty[1], bar_f32_full[FA2_MAX_F32], bar_f32_empty[FA2_MAX_F32];
  __shared__ uint32_t tmem_base_slot;
  constexpr int half = N1 / 2;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int FS = P.n_stages;        // depth of the fp32 TMA staging ring (the bf16 operand ring of k_fused_analysis is gone)
  uint8_t* s_b1 = smem + P.off_b1;
  uint8_t* s_b2 = smem + P.off_b2;
  float* s_scr = reinterpret_cast<float*>(smem + P.off_scratch);

  if (tid == 0) {
    for (int i = 0; i < FA2_X_STAGES; ++i) { mbar_init(&bar_full[i], FA_LOADER_WARPS); mbar_init(&bar_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_d1_full[i], 1); mbar_init(&bar_d1_empty[i], 128); }
    mbar_init(&bar_d2_full[0], 1); mbar_init(&bar_d2_empty[0], 128);
    for (int i = 0; i < FS; ++i) { mbar_init(&bar_f32_full[i], 1); mbar_init(&bar_f32_empty[i], FA_LOADER_WARPS); }
    mbar_init(&bar_b2_full, 128);
    mbar_init(&bar_b2_empty, 1);
    mbar_init_fence();
  }
  if (warp == 8) tmem_alloc(&tmem_base_slot, (uint32_t)P.tmem_cols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  if (warp < FA_LOADER_WARP0) {
    // constant operand images are staged by the consumer-side warps only; the loaders start streaming x at once
    constexpr int NT = FA_LOADER_WARP0 * 32;
    copy_image(s_b1, P.b1_img, (2 * N1 * P.W * 2) / 16, tid, NT);
    if (warp < 4) {   // leading-dim table -> tensor memory: lane = table row, two bf16 K-elements per 32-bit column
      const uint32_t* src = reinterpret_cast<const uint32_t*>(P.a2_img) + (size_t)(warp * 32 + lane) * 128;
      const uint32_t tm_a2_w = tmem_base_slot + (uint32_t)(5 * N1) + ((uint32_t)(warp * 32) << 16);
#pragma unroll 2
      for (int c = 0; c < 128; c += 16) {
        uint32_t w[16];
#pragma unroll
        for (int e = 0; e < 16; e += 4) {
          const uint4 v = __ldg(reinterpret_cast<const uint4*>(src + c + e));
          w[e] = v.x; w[e + 1] = v.y; w[e + 2] = v.z; w[e + 3] = v.w;
        }
        tmem_st16(tm_a2_w + c, w);
      }
      tmem_st_wait();
      tc_fence_before_sync();
    }
    uint4* z = reinterpret_cast<uint4*>(s_b2);   // padding rows of B2 (kx >= KX) stay zero for the whole kernel
    for (int i = tid; i < (N1 * 512) / 16; i += NT) z[i] = make_uint4(0, 0, 0, 0);
    fence_proxy_async_smem();
    asm volatile("bar.sync 2, %0;" ::"n"(NT) : "memory");
  }
  const uint32_t tmem = tmem_base_slot;
  const uint32_t tm_d1[2] = {tmem, tmem + (uint32_t)(2 * N1)};
  // columns: D1[2] 4*N1 | D2 N1 (single) | leading-dim table 128 | x operand ring FA2_X_STAGES x (32 hi + 32 lo)
  const uint32_t tm_d2[1] = {tmem + (uint32_t)(4 * N1)};
  const uint32_t tm_a2 = tmem + (uint32_t)(5 * N1);
  const uint32_t tm_x = tmem + (uint32_t)(5 * N1 + 128);

  const int n_local = (P.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == FA_TMA_WARP) {
    // ------------------------------------------------------------------ TMA producer: one tensor load per 32 KB slab
    const int total = n_local * P.slabs;
    uint8_t* f32_stage = smem + P.off_f32;
    const uint64_t pol = l2_policy_evict_first();
    pdl_wait();                                  // x is produced by the previous kernel of the stream
    // Hand-over to the next kernel of the stream only AFTER this CTA has seen its own predecessor complete: a kernel of this
    // library may then read, ahead of its own wait, anything its immediate predecessor does not write (the contraction
    // fetches the weights that way).  The dependents still start as soon as this CTA leaves its SM.
    pdl_launch_dependents();
    constexpr unsigned long long PF_PIECE = 8192;
    for (int idx = 0; idx < total; ++idx) {
      const int sb = idx % FS;
      mbar_wait(&bar_f32_empty[sb], (uint32_t)(((idx / FS) & 1) ^ 1));
      if (elect_one()) {
#pragma unroll
        for (int r = 0; r < 2; ++r) {        // this CTA's idx-th 8 KB piece of each prefetch range
          const unsigned long long off = ((unsigned long long)idx * gridDim.x + blockIdx.x) * PF_PIECE;
          if (off < P.pf_bytes[r]) {
            const unsigned long long left = P.pf_bytes[r] - off;
            bulk_prefetch_l2(P.pf_ptr[r] + off, (uint32_t)(left < PF_PIECE ? left : PF_PIECE));
          }
        }
        const int tile = (int)blockIdx.x + (idx / P.slabs) * (int)gridDim.x, slab = idx % P.slabs;
        // a slab = two [128 rows x 32 floats] boxes in the 128-byte swizzle: a thread can then read ITS ROW conflict-free
        // (16-bit x: ONE [128 rows x 64 elements] box, same row length and swizzle)
        constexpr int n_boxes = S == 0 ? 2 : 1;
        mbar_arrive_expect_tx(&bar_f32_full[sb], (uint32_t)(n_boxes * 16384));
#pragma unroll
        for (int hb = 0; hb < n_boxes; ++hb) {
          if (P.l2_stream_hint) tma_load_2d_hint(f32_stage + sb * 32768 + hb * 16384, &x_map, &bar_f32_full[sb], slab * 64 + hb * 32, tile * 128, pol);
          else tma_load_2d(f32_stage + sb * 32768 + hb * 16384, &x_map, &bar_f32_full[sb], slab * 64 + hb * 32, tile * 128);
        }
      }
      __syncwarp();
    }
  } else if (warp >= FA_LOADER_WARP0) {
    // ------------------------------------------------------------------ converters: fp32 staging -> bf16 hi / lo -> TENSOR MEMORY
    // The A operand of stage 1 (the image rows) lives in tensor memory: thread <-> image row (its TMEM lane) and one of the two
    // 32-float boxes of the slab.  Versus the shared-memory operand ring of k_fused_analysis this removes, per 128-row tile, the
    // 64 KB of swizzled bf16 stores and the 64 KB the MMAs re-read from them (the kernel is bound by shared-memory bandwidth).
    // (a warp may only touch TMEM lanes 32 * (warp % 4) .. +31: the quarter is warp % 4, NOT the index within the converter group)
    const int cw = warp - FA_LOADER_WARP0, q = warp & 3, hb = cw >> 2;
    const int row = 32 * q + lane;
    uint8_t* f32_stage = smem + P.off_f32;
    const uint32_t my_row = (uint32_t)((S == 0 ? hb * 16384 : 0) + row * 128);
    const uint32_t sw = (uint32_t)(row & 7);
    const uint32_t tm_mine = tm_x + ((uint32_t)(32 * q) << 16) + (uint32_t)(16 * hb);
    const int total = n_local * P.slabs;
    for (int idx = 0; idx < total; ++idx) {
      const int xs = idx % FA2_X_STAGES;
      const int sb = idx % FS;
      if (warp == FA_LOADER_WARP0) SC_TRACE(P, 0, idx, 0);
      mbar_wait(&bar_f32_full[sb], (uint32_t)((idx / FS) & 1));
      if (warp == FA_LOADER_WARP0) SC_TRACE(P, 7, idx, 0);
      uint32_t hi[16], lo[16];
      const uint8_t* fsrc = f32_stage + sb * 32768 + my_row;
      if constexpr (S == 0) {
#pragma unroll
        for (int c = 0; c < 8; ++c) {            // 16-byte chunk c of the row sits at chunk position c ^ (row & 7)
          const float4 v = *reinterpret_cast<const float4*>(fsrc + ((c ^ sw) << 4));
          split2_bf16(v.x, v.y, hi[2 * c], lo[2 * c]);
          split2_bf16(v.z, v.w, hi[2 * c + 1], lo[2 * c + 1]);
        }
      } else {
#pragma unroll
        for (int c = 0; c < 4; ++c) {            // this warp's half of the row: 16-byte chunks 4 hb .. 4 hb + 3, 8 elements each
          const uint4 v = *reinterpret_cast<const uint4*>(fsrc + (((4 * hb + c) ^ sw) << 4));
          const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int e = 0; e < 4; ++e)
            split2_bf16(g16_load<S>((uint16_t)(w[e] & 0xffffu)), g16_load<S>((uint16_t)(w[e] >> 16)), hi[4 * c + e], lo[4 * c + e]);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_f32_empty[sb]);   // this warp has consumed its pieces of the staging buffer
      if (warp == FA_LOADER_WARP0) SC_TRACE(P, 0, idx, 1);
      mbar_wait(&bar_empty[xs], (uint32_t)(((idx / FA2_X_STAGES) & 1) ^ 1));
      tc_fence_after_sync();
      if (warp == FA_LOADER_WARP0) SC_TRACE(P, 0, idx, 2);
      tmem_st16(tm_mine + (uint32_t)(64 * xs), hi);
      tmem_st16(tm_mine + (uint32_t)(64 * xs + 32), lo);
      tmem_st_wait();
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_full[xs]);
    }
  } else if (warp == 8) {
    // ------------------------------------------------------------------ stage-1 MMA issuer (warp-uniform, one elected lane issues)
    {
      const uint32_t idesc_p1 = idesc_bf16(128, 2 * N1), idesc_p2 = idesc_bf16(128, N1);
      const uint32_t b1_lo = desc_lo(smem_u32(s_b1));
      uint32_t g = 0;
      for (int i = 0; i < n_local; ++i) {
        const int buf = i & 1;
        SC_TRACE(P, 1, i, 0);
        mbar_wait(&bar_d1_empty[buf], (uint32_t)(((i >> 1) & 1) ^ 1));
        tc_fence_after_sync();
        SC_TRACE(P, 1, i, 1);
        for (int s = 0; s < P.slabs; ++s, ++g) {
          const int xs = (int)(g % (uint32_t)FA2_X_STAGES);
          mbar_wait(&bar_full[xs], (g / (uint32_t)FA2_X_STAGES) & 1u);
          tc_fence_after_sync();
          const uint32_t x_hi = tm_x + (uint32_t)(64 * xs), x_lo = x_hi + 32;
          const uint32_t d_b = b1_lo + (uint32_t)s * ((2 * N1 * 128) >> 4);
          if (elect_one()) {
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              mma_bf16_ts(tm_d1[buf], x_hi + 8 * kk, desc_from_lo(d_b + 2 * kk), idesc_p1, (s | kk) != 0);
              mma_bf16_ts(tm_d1[buf], x_lo + 8 * kk, desc_from_lo(d_b + 2 * kk), idesc_p2, true);
            }
            mma_commit(&bar_empty[xs]);
          }
          __syncwarp();
        }
        if (elect_one()) mma_commit(&bar_d1_full[buf]);
        __syncwarp();
        SC_TRACE(P, 1, i, 2);
      }
    }
    __syncwarp();
  } else if (warp == 9) {
    // ------------------------------------------------------------------ stage-2 MMA issuer
    {
      const uint32_t idesc_p2 = idesc_bf16(128, N1);
      const uint32_t b2_lo = desc_lo(smem_u32(s_b2));
      for (int i = 0; i < n_local; ++i) {
        const int buf = 0;
        SC_TRACE(P, 3, i, 0);
        mbar_wait(&bar_b2_full, (uint32_t)(i & 1));
        mbar_wait(&bar_d2_empty[buf], (uint32_t)((i & 1) ^ 1));
        tc_fence_after_sync();
        SC_TRACE(P, 3, i, 1);
        if (elect_one()) {
#pragma unroll
          for (int ks = 0; ks < 16; ++ks) {
            const int slab = ks >> 2, kk = ks & 3;
            mma_bf16_ts(tm_d2[buf], tm_a2 + ks * 8, desc_from_lo(b2_lo + slab * ((N1 * 128) >> 4) + 2 * kk), idesc_p2, ks > 0);
          }
          mma_commit(&bar_b2_empty);
          mma_commit(&bar_d2_full[buf]);
        }
        __syncwarp();
        SC_TRACE(P, 3, i, 2);
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ epilogue 1: D1 -> B operand of stage 2
    const int q4 = warp - 4;                                  // TMEM lane quarter; tile row h = q4*32 + lane
    const uint32_t lane_sel = (uint32_t)(q4 * 32) << 16;
    const int KX = P.KX;
    // B2[n][k2], k2 = 2*h + part: row h owns 4 bytes of every row n, inside K-slab q4 (64 columns = 32 rows h)
    uint8_t* b2_mine = s_b2 + q4 * (N1 * 128) + (lane & 3) * 4;
    const int chunk = lane >> 2;
    for (int i = 0; i < n_local; ++i) {
      const int buf = i & 1;
      if (warp == 4) SC_TRACE(P, 2, i, 0);
      mbar_wait(&bar_d1_full[buf], (uint32_t)((i >> 1) & 1));
      mbar_wait(&bar_b2_empty, (uint32_t)((i & 1) ^ 1));
      tc_fence_after_sync();
      if (warp == 4) SC_TRACE(P, 2, i, 1);
#pragma unroll
      for (int c = 0; c < N1; c += 16) {
        float t1[16], t2[16];
        tmem_ld16(tm_d1[buf] + lane_sel + c, t1);        // x_hi*T1 + x_lo*T1
        tmem_ld16(tm_d1[buf] + lane_sel + N1 + c, t2);   // x_hi*T2
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int kx = c / 2 + e;                       // compile-time; slots kx >= KX hold exact zeros (zero table rows)
          uint32_t hi, lo;
          split2_bf16(t1[2 * e] + t2[2 * e], t1[2 * e + 1] + t2[2 * e + 1], hi, lo);
          *reinterpret_cast<uint32_t*>(b2_mine + kx * 128 + ((chunk ^ (kx & 7)) << 4)) = hi;
          *reinterpret_cast<uint32_t*>(b2_mine + (half + kx) * 128 + ((chunk ^ ((half + kx) & 7)) << 4)) = lo;
        }
      }
      tc_fence_before_sync();
      mbar_arrive(&bar_d1_empty[buf]);
      fence_proxy_async_smem();
      mbar_arrive(&bar_b2_full);
      if (warp == 4) SC_TRACE(P, 2, i, 2);
    }
  } else {
    // ------------------------------------------------------------------ epilogue 2: D2 -> kept modes
    const int row = warp * 32 + lane;                        // output row i' (0-63: T1 rows, 64-127: T2 rows)
    const uint32_t lane_sel = (uint32_t)(warp * 32) << 16;
    const int KX = P.KX;
    pdl_wait();                                              // the mode buffer may still be read by the previous kernel
    for (int i = 0; i < n_local; ++i) {
      const int buf = 0;
      if (warp == 0) SC_TRACE(P, 4, i, 0);
      mbar_wait(&bar_d2_full[buf], (uint32_t)(i & 1));
      tc_fence_after_sync();
      if (warp == 0) SC_TRACE(P, 4, i, 1);
      float d[N1];
#pragma unroll
      for (int c = 0; c < N1; c += 16) tmem_ld16(tm_d2[buf] + lane_sel + c, *reinterpret_cast<float(*)[16]>(&d[c]));
      tmem_ld_wait();
      if (warp == 0) SC_TRACE(P, 5, i, 0);
      tc_fence_before_sync();
      mbar_arrive(&bar_d2_empty[buf]);
      if (warp == 0) SC_TRACE(P, 5, i, 1);
      // T2 rows (warps 2,3) hand hi+lo sums to the matching T1 rows (warps 0,1).  Straight-line code over all N1/2 column
      // slots (padding slots carry exact zeros): runtime bounds checks here turn into a serial LDS->FADD->SHFL->STS chain.
      constexpr int SP = half + 1;                 // scratch row pitch in floats
      if (warp >= 2) {
        float* dst = s_scr + (row - 64) * SP;
#pragma unroll
        for (int kx = 0; kx < half; ++kx) dst[kx] = d[kx] + d[half + kx];
      }
      if (tid == 0) bulk_wait_read_1();            // the block stored two tiles ago has left its staging buffer
      if (warp == 0) SC_TRACE(P, 5, i, 2);
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (warp == 0) SC_TRACE(P, 6, i, 0);
      // the tile's modes are ONE contiguous block of QROWS*KX complex numbers: stage it, then a single bulk async store
      float2* stage = reinterpret_cast<float2*>(smem + P.off_scratch + P.stage_off) + (i & 1) * (P.QROWS * KX);
      if (warp < 2) {
        const float* src = s_scr + row * SP;
        const int q = row >> 1, part = row & 1;
        const bool live = q < P.QROWS && part == 0;
        float mine[half], other[half];
#pragma unroll
        for (int kx = 0; kx < half; ++kx) mine[kx] = d[kx] + d[half + kx] + src[kx];
#pragma unroll
        for (int kx = 0; kx < half; ++kx) other[kx] = __shfl_xor_sync(0xffffffffu, mine[kx], 1);
        float2* my = stage + q * KX;
#pragma unroll
        for (int kx = 0; kx < half; ++kx)
          if (live && kx < KX) my[kx] = make_float2(mine[kx], other[kx]);
      }
      if (warp == 0) SC_TRACE(P, 6, i, 1);
      fence_proxy_async_smem();
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (warp == 0) SC_TRACE(P, 6, i, 2);
      if (P.quad_major && P.qm_tma) {
        // the tile's modes [quad][8 floats] go out as ONE tensor store (box {8 floats, 1 image, Mt/4 quads}): the TMA engine scatters
        // the 32-byte sectors asynchronously (the per-thread store loop below cost ~1500 of this role's ~2700 cycles per tile)
        if (tid == 0) {
          const int tile = (int)blockIdx.x + i * (int)gridDim.x;
          tma_store_3d(&qm_map, stage, 0, tile, 0);
          bulk_commit();
        }
      } else if (P.quad_major) {
        // one 32-byte sector per (image of the tile, quad of modes): element (image, m) lives at ((m >> 2) * n_images + image) * 4 + (m & 3)
        const int tile = (int)blockIdx.x + i * (int)gridDim.x;
        const int nq = P.Mt >> 2;
        for (int idx = tid; idx < P.G * nq; idx += 128) {
          const int g = idx / nq, q = idx - g * nq;
          const float4* sp = reinterpret_cast<const float4*>(stage + g * P.Mt + 4 * q);
          const float4 lo4 = sp[0], hi4 = sp[1];
          const float o8[8] = {lo4.x, lo4.y, lo4.z, lo4.w, hi4.x, hi4.y, hi4.z, hi4.w};
          st_global_v8(reinterpret_cast<float*>(P.out + ((long long)q * P.n_images + (long long)tile * P.G + g) * 4), o8);
        }
      } else if (tid == 0) {
        const int tile = (int)blockIdx.x + i * (int)gridDim.x;
        bulk_store(P.out + (size_t)tile * P.QROWS * KX, stage, (uint32_t)(P.QROWS * KX * 8));
        bulk_commit();
      }
      if (warp == 0) SC_TRACE(P, 4, i, 2);
    }
    if (tid == 0) bulk_wait_all();
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 8) tmem_dealloc(tmem, (uint32_t)P.tmem_cols);
}

// =====================================================================================================
// fused synthesis:  kept modes of the G images of a tile  ->  128 image rows (+ bias)
//
//   stage A (leading dim) DA[hl, n] = sum_k AA[hl, k] * BA[n, k]      M=128 (rows)  N=2*N1  K=128 (T1 | T2 halves)
//   stage B (last dim)    DB[hl, w] = sum_j U[hl, j] * TS[j, w]       M=128         N=W     K=N1 x 3 bf16 products
//
//   warps 10-13 prep       modes (standard or quad-major layout) -> bf16 hi/lo real-embedded B operand of stage A (BA[2])
//   warp  8     stage-A MMA issuer (+ TMEM allocation)   BA -> DA[2]
//   warps 4-7   epilogue A: DA -> U -> bf16 hi/lo A operand of stage B (U[2])
//   warp  9     stage-B MMA issuer                        U -> DB[2]
//   warps 0-3, 14-17  epilogue B (two warps per TMEM lane quarter, half of the columns each): DB -> + bias -> swizzled
//               [32 rows x 128 B] box -> one TMA tensor store per box
// =====================================================================================================
constexpr int FS_THREADS = 18 * 32;             // warps 14-17: second epilogue-B group (the other half of the columns)
constexpr int FS_EPI_B_WARPS = 8;
constexpr int FS_STAGE_BYTES = FS_EPI_B_WARPS * 4096;   // per epilogue-B warp one [32 rows x 32 floats] TMA store box

struct SynParams {
  const float2* modes;
  float* out;
  const float* bias;       // may be null
  const uint8_t* aa_img;   // [128 x 128] bf16 image: leading-dim table, columns (2q+s | 64+2q+s)
  const uint8_t* bb_img;   // two [W x 64] bf16 images: T1 then T2 of the last-dim table (rows = w, K = j)
  int n_tiles, W, KX, QROWS, H, n_channels, tmem_cols;
  int l2_stream_hint;      // 1: the image rows are stored with an L2 evict-first policy (written once, not re-read by this step)
  int slices_per_image;    // 3-D: the fused kernel sees (image, z) slices; bias channel = (slice / slices_per_image) % n_channels
  int quad_major, KY;      // 1: the modes arrive in the quad-major layout modes[quad][image][4 modes] (see AnaParams)
  long long n_images;
  uint32_t off_aa, off_ba, off_u, off_bb, off_stage;
  long long* trace;        // debug timeline of CTA 0 (SC_TRACE_FILE), else nullptr
};

// S: storage of the output -- 0 float, SC_FLAG_GRID_F16 / SC_FLAG_GRID_BF16 (only the adjoint synthesis, dx, is launched so): the
// epilogue rounds to nearest even and stores [32 rows x 32 elements] boxes of 64-byte rows in the 64-byte swizzle
template <int N1, int S>
__global__ void __launch_bounds__(FS_THREADS, 1) k_fused_synthesis(const SynParams P, const __grid_constant__ CUtensorMap out_map) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ uint64_t bar_ba_full[2], bar_ba_empty[2], bar_da_full[2], bar_da_empty[2];
  __shared__ uint64_t bar_u_full[2], bar_u_empty[2], bar_db_full[2], bar_db_empty[2];
  __shared__ uint32_t tmem_base_slot;
  constexpr int BA_BYTES = 2 * N1 * 256;      // [2*N1 x 128] bf16 = two slabs of 2*N1 rows
  constexpr int U_BYTES = 2 * FA_SLAB_BYTES;  // hi slab + lo slab, [128 x 64] bf16 each

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int W = P.W, KX = P.KX;
  uint8_t* s_aa = smem + P.off_aa;
  uint8_t* s_ba = smem + P.off_ba;
  uint8_t* s_u = smem + P.off_u;
  uint8_t* s_bb = smem + P.off_bb;

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bar_ba_full[i], 4);  mbar_init(&bar_ba_empty[i], 1);
      mbar_init(&bar_da_full[i], 1);  mbar_init(&bar_da_empty[i], 128);
      mbar_init(&bar_u_full[i], 128); mbar_init(&bar_u_empty[i], 1);
      mbar_init(&bar_db_full[i], 1);  mbar_init(&bar_db_empty[i], 32 * FS_EPI_B_WARPS);
    }
    mbar_init_fence();
  }
  if (warp == 8) tmem_alloc(&tmem_base_slot, (uint32_t)P.tmem_cols);
  copy_image(s_aa, P.aa_img, (128 * 128 * 2) / 16, tid, FS_THREADS);
  copy_image(s_bb, P.bb_img, (2 * W * 128) / 16, tid, FS_THREADS);
  {
    uint4* z1 = reinterpret_cast<uint4*>(s_ba);     // zero both BA buffers and both U buffers once: padding rows /
    for (int i = tid; i < (2 * BA_BYTES) / 16; i += FS_THREADS) z1[i] = make_uint4(0, 0, 0, 0);   // columns stay zero
    uint4* z2 = reinterpret_cast<uint4*>(s_u);
    for (int i = tid; i < (2 * U_BYTES) / 16; i += FS_THREADS) z2[i] = make_uint4(0, 0, 0, 0);
  }
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = tmem_base_slot;
  const uint32_t tm_da[2] = {tmem, tmem + (uint32_t)(2 * N1)};
  const uint32_t tm_db[2] = {tmem + (uint32_t)(4 * N1), tmem + (uint32_t)(4 * N1 + W)};
  const int n_local = (P.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp >= 10 && warp < 14) {
    // ------------------------------------------------------------------ prep: modes -> BA
    // thread -> fixed mode row q (0..31) and columns kx = kx0 + 4u: every swizzled store address is a per-thread base plus
    // a compile-time multiple of 1024 bytes (8 operand rows), so the per-element work is one 8-byte load, one split, six stores
    const int pt = tid - 10 * 32;   // 0..127
    const int q = pt >> 2, kx0 = pt & 3;
    const bool q_ok = q < P.QROWS;
    const uint32_t o_re = sw128_offset(2 * kx0, 2 * q, 2 * N1), o_im = sw128_offset(2 * kx0 + 1, 2 * q, 2 * N1);
    constexpr uint32_t T2 = 2 * N1 * 128;    // second K-slab (columns 64 + k): hi * T2
    constexpr uint32_t LO = N1 * 128;        // rows N1 + n: lo * T1
    pdl_wait();                              // the modes are produced by the previous kernel of the stream
    pdl_launch_dependents();                 // (after the wait: see k_fused_analysis)
    for (int i = 0; i < n_local; ++i) {
      const int buf = i & 1;
      const int tile = (int)blockIdx.x + i * (int)gridDim.x;
      const float2* src = P.modes + ((size_t)tile * P.QROWS + q) * KX + kx0;
      long long ustep = 4;
      if (P.quad_major) {
        const int g = q / P.KY, mbase = (q - g * P.KY) * KX + kx0;      // image of the tile, first mode of this thread's column set
        src = P.modes + ((long long)(mbase >> 2) * P.n_images + (long long)tile * (P.QROWS / P.KY) + g) * 4 + (mbase & 3);
        ustep = P.n_images * 4;
      }
      float2 y[8];
      if (warp == 10) SC_TRACE(P, 0, i, 0);
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (q_ok && kx0 + 4 * u < KX) y[u] = __ldg(src + u * ustep);
      mbar_wait(&bar_ba_empty[buf], (uint32_t)(((i >> 1) & 1) ^ 1));
      if (warp == 10) SC_TRACE(P, 0, i, 1);
      uint8_t* ba = s_ba + buf * BA_BYTES;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (q_ok && kx0 + 4 * u < KX) {
          uint32_t hi, lo;                         // (re | im << 16)
          split2_bf16(y[u].x, y[u].y, hi, lo);
          const uint32_t re_row_hi = hi ^ 0x80000000u, im_row_hi = __byte_perm(hi, 0, 0x1032);   // (re, -im) ; (im, re)
          const uint32_t re_row_lo = lo ^ 0x80000000u, im_row_lo = __byte_perm(lo, 0, 0x1032);
          uint8_t* pr = ba + o_re + u * 1024;      // rows 2*kx advance by 8 per u
          uint8_t* pi = ba + o_im + u * 1024;
          *reinterpret_cast<uint32_t*>(pr) = re_row_hi;             // hi * T1
          *reinterpret_cast<uint32_t*>(pi) = im_row_hi;
          *reinterpret_cast<uint32_t*>(pr + T2) = re_row_hi;        // hi * T2
          *reinterpret_cast<uint32_t*>(pi + T2) = im_row_hi;
          *reinterpret_cast<uint32_t*>(pr + LO) = re_row_lo;        // lo * T1
          *reinterpret_cast<uint32_t*>(pi + LO) = im_row_lo;
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_ba_full[buf]);
      if (warp == 10) SC_TRACE(P, 0, i, 2);
    }
  } else if (warp == 8) {
    // ------------------------------------------------------------------ stage-A MMA issuer
    {
      const uint32_t idesc_a = idesc_bf16(128, 2 * N1);
      const uint32_t aa_lo = desc_lo(smem_u32(s_aa)), ba_lo0 = desc_lo(smem_u32(s_ba));
      for (int i = 0; i < n_local; ++i) {
        const int buf = i & 1;
        const uint32_t ph = (uint32_t)((i >> 1) & 1);
        SC_TRACE(P, 1, i, 0);
        mbar_wait(&bar_ba_full[buf], ph);
        mbar_wait(&bar_da_empty[buf], ph ^ 1u);
        tc_fence_after_sync();
        SC_TRACE(P, 1, i, 1);
        const uint32_t ba_lo = ba_lo0 + (uint32_t)buf * (BA_BYTES >> 4);
        if (elect_one()) {
#pragma unroll
          for (int ks = 0; ks < 8; ++ks) {
            const int slab = ks >> 2, kk = ks & 3;
            mma_bf16_ss(tm_da[buf], desc_from_lo(aa_lo + slab * ((128 * 128) >> 4) + 2 * kk),
                        desc_from_lo(ba_lo + slab * ((2 * N1 * 128) >> 4) + 2 * kk), idesc_a, ks > 0);
          }
          mma_commit(&bar_ba_empty[buf]);
          mma_commit(&bar_da_full[buf]);
        }
        __syncwarp();
        SC_TRACE(P, 1, i, 2);
      }
    }
    __syncwarp();
  } else if (warp == 9) {
    // ------------------------------------------------------------------ stage-B MMA issuer
    {
      const uint32_t idesc_b = idesc_bf16(128, W);
      const uint32_t u_lo0 = desc_lo(smem_u32(s_u));
      const uint32_t t1 = desc_lo(smem_u32(s_bb)), t2 = t1 + (((uint32_t)W * 128) >> 4);
      for (int i = 0; i < n_local; ++i) {
        const int buf = i & 1;
        const uint32_t ph = (uint32_t)((i >> 1) & 1);
        SC_TRACE(P, 3, i, 0);
        mbar_wait(&bar_u_full[buf], ph);
        mbar_wait(&bar_db_empty[buf], ph ^ 1u);
        tc_fence_after_sync();
        SC_TRACE(P, 3, i, 1);
        const uint32_t u_hi = u_lo0 + (uint32_t)buf * (U_BYTES >> 4), u_lo = u_hi + (FA_SLAB_BYTES >> 4);
        if (elect_one()) {
#pragma unroll
          for (int ks = 0; ks < N1 / 16; ++ks) {
            mma_bf16_ss(tm_db[buf], desc_from_lo(u_hi + 2 * ks), desc_from_lo(t1 + 2 * ks), idesc_b, ks > 0);
            mma_bf16_ss(tm_db[buf], desc_from_lo(u_lo + 2 * ks), desc_from_lo(t1 + 2 * ks), idesc_b, true);
            mma_bf16_ss(tm_db[buf], desc_from_lo(u_hi + 2 * ks), desc_from_lo(t2 + 2 * ks), idesc_b, true);
          }
          mma_commit(&bar_u_empty[buf]);
          mma_commit(&bar_db_full[buf]);
        }
        __syncwarp();
        SC_TRACE(P, 3, i, 2);
      }
    }
    __syncwarp();
  } else if (warp >= 4 && warp < 8) {
    // ------------------------------------------------------------------ epilogue A: DA -> U (hi / lo)
    const int q4 = warp - 4;
    const int row = q4 * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q4 * 32) << 16;
    for (int i = 0; i < n_local; ++i) {
      const int buf = i & 1;
      const uint32_t ph = (uint32_t)((i >> 1) & 1);
      if (warp == 4) SC_TRACE(P, 2, i, 0);
      mbar_wait(&bar_da_full[buf], ph);
      mbar_wait(&bar_u_empty[buf], ph ^ 1u);
      tc_fence_after_sync();
      if (warp == 4) SC_TRACE(P, 2, i, 1);
      uint8_t* uhi = s_u + buf * U_BYTES + row * 128;
      uint8_t* ulo = uhi + FA_SLAB_BYTES;
#pragma unroll
      for (int c = 0; c < N1; c += 32) {            // two 16-column chunks (4 TMEM loads) per wait
        float t1[2][16], t2[2][16];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          if (c + 16 * h < N1) {
            tmem_ld16(tm_da[buf] + lane_sel + c + 16 * h, t1[h]);
            tmem_ld16(tm_da[buf] + lane_sel + N1 + c + 16 * h, t2[h]);
          }
        }
        tmem_ld_wait();
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          if (c + 16 * h < N1) {
            uint32_t hw[8], lw[8];
#pragma unroll
            for (int e = 0; e < 8; ++e)
              split2_bf16(t1[h][2 * e] + t2[h][2 * e], t1[h][2 * e + 1] + t2[h][2 * e + 1], hw[e], lw[e]);
            const int c0 = (c + 16 * h) / 8;          // two 16-byte chunks of 8 consecutive j
            *reinterpret_cast<uint4*>(uhi + (((c0 ^ row) & 7) << 4)) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
            *reinterpret_cast<uint4*>(uhi + ((((c0 + 1) ^ row) & 7) << 4)) = make_uint4(hw[4], hw[5], hw[6], hw[7]);
            *reinterpret_cast<uint4*>(ulo + (((c0 ^ row) & 7) << 4)) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
            *reinterpret_cast<uint4*>(ulo + ((((c0 + 1) ^ row) & 7) << 4)) = make_uint4(lw[4], lw[5], lw[6], lw[7]);
          }
        }
      }
      tc_fence_before_sync();
      mbar_arrive(&bar_da_empty[buf]);
      fence_proxy_async_smem();
      mbar_arrive(&bar_u_full[buf]);
      if (warp == 4) SC_TRACE(P, 2, i, 2);
    }
  } else {
    // ------------------------------------------------------------------ epilogue B (warps 0-3 and 14-17): DB -> image rows
    // Two warps per TMEM lane quarter, each taking half of the columns: the store side of a tile (TMEM -> registers -> +bias ->
    // swizzled box -> TMA tensor store) was the longest role of the pipeline with four warps (measured write rate 3.9 TB/s
    // against 7.5 TB/s for a plain fill on the same GPU).
    const int q = warp & 3;                 // a warp may only touch TMEM lanes 32 * (warp % 4) ..: warps 14-17 -> quarters 2, 3, 0, 1
    const int hb = warp < 4 ? 0 : 1;
    const int row = q * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    uint8_t* box = smem + P.off_stage + (hb * 4 + q) * 4096;   // one [32 x 128 B] box per warp
    const int c_begin = hb * (W / 2), c_end = c_begin + W / 2;
    const uint64_t pol = l2_policy_evict_first();
    pdl_wait();                                             // the output image may still be read by the previous kernel
    for (int i = 0; i < n_local; ++i) {
      const int buf = i & 1;
      const uint32_t ph = (uint32_t)((i >> 1) & 1);
      const int tile = (int)blockIdx.x + i * (int)gridDim.x;
      float b = 0.f;
      if (P.bias != nullptr) {
        const long long slice = (long long)tile * (128 / P.H) + row / P.H;
        b = __ldg(P.bias + (int)((slice / P.slices_per_image) % P.n_channels));
      }
      if (warp == 0) SC_TRACE(P, 4, i, 0);
      mbar_wait(&bar_db_full[buf], ph);
      tc_fence_after_sync();
      if (warp == 0) SC_TRACE(P, 4, i, 1);
      // 32 columns at a time: TMEM -> registers (+bias) -> this warp's [32 rows x 128 B] staging box in the tensor map's
      // 128-byte swizzle -> ONE TMA tensor store per warp and box (direct per-thread row stores touch 32 different
      // 128-byte lines per warp instruction and serialise in the LSU).
      for (int c = c_begin; c < c_end; c += 32) {
        float t[2][16];
        tmem_ld16(tm_db[buf] + lane_sel + c, t[0]);
        tmem_ld16(tm_db[buf] + lane_sel + c + 16, t[1]);
        if (lane == 0) bulk_wait_read();            // the previous store of this warp has finished reading the box
        __syncwarp();
        tmem_ld_wait();
        if constexpr (S == 0) {
#pragma unroll
          for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int e = 0; e < 16; e += 4) {
              const int ch = (16 * u + e) >> 2;        // 16-byte chunk index within the 128-byte row
              *reinterpret_cast<float4*>(box + lane * 128 + (((ch ^ lane) & 7) << 4)) =
                  make_float4(t[u][e] + b, t[u][e + 1] + b, t[u][e + 2] + b, t[u][e + 3] + b);
            }
        } else {
#pragma unroll
          for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int e = 0; e < 16; e += 8) {
              const int ch = (16 * u + e) >> 3;        // 16-byte chunk (8 elements) within the 64-byte row; 64-byte swizzle
              *reinterpret_cast<uint4*>(box + lane * 64 + (((ch ^ (lane >> 1)) & 3) << 4)) =
                  make_uint4(g16_pack2<S>(t[u][e] + b, t[u][e + 1] + b), g16_pack2<S>(t[u][e + 2] + b, t[u][e + 3] + b),
                             g16_pack2<S>(t[u][e + 4] + b, t[u][e + 5] + b), g16_pack2<S>(t[u][e + 6] + b, t[u][e + 7] + b));
            }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          if (P.l2_stream_hint) tma_store_2d_hint(&out_map, box, c, tile * 128 + q * 32, pol);
          else
            tma_store_2d(&out_map, box, c, tile * 128 + q * 32);
          bulk_commit();
        }
      }
      tc_fence_before_sync();
      mbar_arrive(&bar_db_empty[buf]);
      if (warp == 0) SC_TRACE(P, 4, i, 2);
    }
    if (lane == 0) bulk_wait_all();
    __syncwarp();
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 8) tmem_dealloc(tmem, (uint32_t)P.tmem_cols);
}

// =====================================================================================================
// mode-wise complex GEMM on tcgen05 (dense contraction and its two backward products)
//
//   out[R, n] = sum_k a(R, k) * b(n, k)   (complex), one independent product per kept mode m.
//   The complex product is a real GEMM with the 2x2 embedding on the A side:
//     rows (R, re|im) x K (k, re|im):   [ ar  -ai ]        B rows n, K (k, re|im) = (br, bi) as stored
//                                       [ ai   ar ]
//   A = A_hi + A_lo and B = B_hi + B_lo in bf16; D = A_hi*[B_hi ; B_lo] + A_lo*B_hi  (FP32 in TMEM).
//   warps 0-3 epilogue, warp 4 MMA issuer (+TMEM), warps 5-20 gather/split loaders.
//   A CTA owns a CONTIGUOUS range of modes: the 8-byte gathers of 4 consecutive modes share 32-byte sectors, so the
//   sectors fetched for the first mode of a range are L2 hits for the next three.
// =====================================================================================================
constexpr int MG2_LOADER_WARPS = 16;
constexpr int MG2_THREADS = (5 + MG2_LOADER_WARPS) * 32;
constexpr int MG2_LOADERS = MG2_LOADER_WARPS * 32;

struct ModeGemmTcParams {
  const float2* a; const float2* b; float2* out;
  long long sAR, sAK, sBN, sBK, sOR, sON;          // complex-element strides
  const int* offA; const int* offB; const int* offO;   // per-mode offsets (nullptr -> m)
  int MR, NB, KC;                                   // complex rows of A (<= 64), rows of B (<= 64), contraction length
  int NBp;                                          // NB rounded up to a multiple of 16
  int Kreal;                                        // 2 * KC rounded up to a multiple of 64
  int KCp, kshift;                                  // KC rounded up to a power of two (>= 8), and its log2
  int conjA;
  int n_modes, modes_per_cta;
  uint32_t stage_bytes, off_alo, off_b;
};

__global__ void __launch_bounds__(MG2_THREADS, 1) k_mode_gemm_tc(const ModeGemmTcParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ uint64_t bar_full[2], bar_empty[2], bar_d_full[2], bar_d_empty[2];
  __shared__ uint32_t tmem_base_slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bar_full[i], MG2_LOADER_WARPS); mbar_init(&bar_empty[i], 1);
      mbar_init(&bar_d_full[i], 1); mbar_init(&bar_d_empty[i], 128);
    }
    mbar_init_fence();
  }
  if (warp == 4) tmem_alloc(&tmem_base_slot, 256);
  {
    uint4* z = reinterpret_cast<uint4*>(smem);      // padding rows / columns of both stages stay zero
    for (int i = tid; i < (int)(2 * P.stage_bytes / 16); i += MG2_THREADS) z[i] = make_uint4(0, 0, 0, 0);
  }
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = tmem_base_slot;
  const int m_begin = (int)blockIdx.x * P.modes_per_cta;
  const int n_local = min(P.modes_per_cta, P.n_modes - m_begin);
  const int rowsB = 2 * P.NBp;

  if (warp >= 5) {
    // ------------------------------------------------------------------ gather + split loaders
    // thread -> fixed contraction index k, rows r0, r0 + step, ...: all index math is hoisted out of the mode loop and the
    // per-element work is one 8-byte gather, one bf16 hi/lo split and four (A) / two (B) 4-byte swizzled stores.
    const int lt = tid - 5 * 32;
    const int k = lt & (P.KCp - 1);
    const int r0 = lt >> P.kshift;
    const int step = MG2_LOADERS >> P.kshift;          // 8, 16, 32 or 64 rows between a thread's elements
    const bool k_ok = k < P.KC;
    const long long a_elem0 = (long long)r0 * P.sAR + (long long)k * P.sAK, a_estep = (long long)step * P.sAR;
    const long long b_elem0 = (long long)r0 * P.sBN + (long long)k * P.sBK, b_estep = (long long)step * P.sBN;
    // step is a multiple of 8, so (row & 7) -- the swizzle phase -- is the same for all of a thread's rows
    const uint32_t a_s0 = sw128_offset(2 * r0, 2 * k, 128), a_s1 = sw128_offset(2 * r0 + 1, 2 * k, 128);
    const uint32_t a_sstep = (uint32_t)step * 256u;
    const uint32_t b_s0 = sw128_offset(r0, 2 * k, rowsB), b_sstep = (uint32_t)step * 128u, b_lo = (uint32_t)P.NBp * 128u;
    for (int it = 0; it < n_local; ++it) {
      const int m = m_begin + it;
      const int st = it & 1;
      const float2* pa = P.a + (P.offA ? (long long)__ldg(P.offA + m) : (long long)m) + a_elem0;
      const float2* pb = P.b + (P.offB ? (long long)__ldg(P.offB + m) : (long long)m) + b_elem0;
      uint8_t* a_hi = smem + (size_t)st * P.stage_bytes;
      uint8_t* a_lo = a_hi + P.off_alo;
      uint8_t* b_op = a_hi + P.off_b;
      float2 v[8], w[8];
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (k_ok && r0 + u * step < P.MR) v[u] = __ldg(pa + u * a_estep);
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (k_ok && r0 + u * step < P.NB) w[u] = __ldg(pb + u * b_estep);
      mbar_wait(&bar_empty[st], (uint32_t)(((it >> 1) & 1) ^ 1));
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (k_ok && r0 + u * step < P.MR) {
          uint32_t hi, lo;
          split2_bf16(v[u].x, v[u].y, hi, lo);                 // (re | im << 16)
          uint32_t r0h, r1h, r0l, r1l;
          if (P.conjA) {   // a = conj(v): row re = (vr, vi), row im = (-vi, vr)
            r0h = hi; r1h = __byte_perm(hi, 0, 0x1032) ^ 0x00008000u;
            r0l = lo; r1l = __byte_perm(lo, 0, 0x1032) ^ 0x00008000u;
          } else {         // a = v:       row re = (vr, -vi), row im = (vi, vr)
            r0h = hi ^ 0x80000000u; r1h = __byte_perm(hi, 0, 0x1032);
            r0l = lo ^ 0x80000000u; r1l = __byte_perm(lo, 0, 0x1032);
          }
          *reinterpret_cast<uint32_t*>(a_hi + a_s0 + u * a_sstep) = r0h;
          *reinterpret_cast<uint32_t*>(a_hi + a_s1 + u * a_sstep) = r1h;
          *reinterpret_cast<uint32_t*>(a_lo + a_s0 + u * a_sstep) = r0l;
          *reinterpret_cast<uint32_t*>(a_lo + a_s1 + u * a_sstep) = r1l;
        }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (k_ok && r0 + u * step < P.NB) {
          uint32_t hi, lo;
          split2_bf16(w[u].x, w[u].y, hi, lo);
          *reinterpret_cast<uint32_t*>(b_op + b_s0 + u * b_sstep) = hi;          // row n        (hi)
          *reinterpret_cast<uint32_t*>(b_op + b_s0 + u * b_sstep + b_lo) = lo;   // row NBp + n  (lo)
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_full[st]);
    }
  } else if (warp == 4) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      const uint32_t idesc1 = idesc_bf16(128, rowsB), idesc2 = idesc_bf16(128, P.NBp);
      for (int it = 0; it < n_local; ++it) {
        const int st = it & 1;
        const uint32_t ph = (uint32_t)((it >> 1) & 1);
        mbar_wait(&bar_full[st], ph);
        mbar_wait(&bar_d_empty[st], ph ^ 1u);
        tc_fence_after_sync();
        const uint32_t a_hi = desc_lo(smem_u32(smem + (size_t)st * P.stage_bytes)), a_lo = a_hi + (P.off_alo >> 4),
                       b_op = a_hi + (P.off_b >> 4);
        const uint32_t d = tmem + (uint32_t)(st * 128);
        const int slabs = P.Kreal / 64;
        for (int slab = 0; slab < slabs; ++slab) {
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            const uint64_t db = desc_from_lo(b_op + slab * ((rowsB * 128) >> 4) + 2 * kk);
            mma_bf16_ss(d, desc_from_lo(a_hi + slab * ((128 * 128) >> 4) + 2 * kk), db, idesc1, (slab | kk) != 0);
            mma_bf16_ss(d, desc_from_lo(a_lo + slab * ((128 * 128) >> 4) + 2 * kk), db, idesc2, true);
          }
        }
        mma_commit(&bar_empty[st]);
        mma_commit(&bar_d_full[st]);
      }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------------ epilogue
    const int row = warp * 32 + lane;                // real row (R, part)
    const int R = row >> 1, part = row & 1;
    const uint32_t lane_sel = (uint32_t)(warp * 32) << 16;
    for (int it = 0; it < n_local; ++it) {
      const int m = m_begin + it;
      const int st = it & 1;
      const long long mo = P.offO ? (long long)__ldg(P.offO + m) : m;
      mbar_wait(&bar_d_full[st], (uint32_t)((it >> 1) & 1));
      tc_fence_after_sync();
      const uint32_t d = tmem + (uint32_t)(st * 128) + lane_sel;
      float2* dst = P.out + mo + (long long)R * P.sOR;
      for (int c = 0; c < P.NBp; c += 8) {           // hi block [0, NBp), lo block [NBp, 2*NBp)
        float t1[8], t2[8];
        tmem_ld8(d + c, t1);
        tmem_ld8(d + P.NBp + c, t2);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int n = c + e;
          const float mine = t1[e] + t2[e];
          const float other = __shfl_xor_sync(0xffffffffu, mine, 1);
          if (part == 0 && R < P.MR && n < P.NB) dst[(long long)n * P.sON] = make_float2(mine, other);
        }
      }
      tc_fence_before_sync();
      mbar_arrive(&bar_d_empty[st]);
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem, 256);
}

// helpers of the quad kernels below (four consecutive modes of one element = one aligned 32-byte sector)
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ void ld_global_v8(const float2* p, float (&v)[8]) {
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
               : "l"(p));
}

// per-role clock64 timeline of CTA 0 of the quad kernels, only in -DSC_TRACE_QUAD builds (scripts/trace_run.py)
#ifdef SC_TRACE_QUAD
#define SC_QTRACE(P, role, i, ph) SC_TRACE(P, role, i, ph)
#else
#define SC_QTRACE(P, role, i, ph) do { } while (0)
#endif

// =====================================================================================================
// mode-wise complex GEMM, four consecutive modes per CTA, second generation ("quad2")
//
//   Sector-exact global traffic (one 256-bit load / store per 4 modes of an element) like the round-1 quad kernel it replaced
//   (that one kept both operands as bf16 tiles in shared memory, 192 KB, and consumed K in two serial rounds); here:
//     * the A operand (2x2-embedded, bf16 hi / lo) lives in TENSOR MEMORY: the loader thread that owns real row r converts
//       its row's values in registers and writes them with tcgen05.st into a 4-slot ring of 8-k chunks (one MMA K-step);
//     * the B operand (as stored, bf16 hi rows / lo rows) is the only shared-memory operand: K-slabs of 32 complex k,
//       3-slot ring (never recycled for K <= 96);
//     * ONE accumulator per mode: D += A_hi*B_hi + A_hi*B_lo + A_lo*B_hi as three N = NBp MMAs per K-step (hi / lo products
//       in separate columns would take twice the tensor memory);
//     * loads are software-pipelined two batches deep per thread with L2 prefetches ahead of them, and operands that the
//       previous kernel of the stream does not write (weights, saved modes) are fetched BEFORE the grid-dependency wait.
//   Any MR / NB / KC: 64-row and 64-column tiles over gridDim.y, K streamed through the rings.
//   warp 0 MMA issue (+TMEM), warp 1 dependency hand-over (+ fused bias gradient), warps 4-11 A loaders, 12-19 B loaders,
//   all 20 warps epilogue.
// =====================================================================================================
constexpr int MQ2_A_WARPS = 8, MQ2_B_WARPS = 8;
constexpr int MQ2_THREADS = (4 + MQ2_A_WARPS + MQ2_B_WARPS) * 32;   // 640
constexpr int MQ2_A_SLOTS = 4;                  // TMEM ring: per slot 4 modes x (8 hi + 8 lo) columns
constexpr int MQ2_B_SLOTS = 3;                  // shared-memory ring of K-slabs
constexpr uint32_t MQ2_SLAB_BYTES = 65536;      // one K-slab of B for 4 modes
constexpr uint32_t MQ2_MODE_BYTES = 16384;      // [<= 128 rows (hi, lo) x 128 B]
constexpr uint32_t MQ2_TM_A = 256;              // D of mode j at column 64 j; A slot s at 256 + 64 s (+16 j, lo +8)

struct ModeGemmQuad2Params {
  const float2* a; const float2* b; float2* out;
  long long sAR, sAK, sBN, sBK, sOR, sON;       // complex-element strides
  long long sAQ, sBQ, sOQ;                      // stride between quads: 4 in the standard (.., modes) layout; the quad-major layout
                                                // [quad][..][4 modes] of the internal mode tensors has its own (see sc_api.cu)
  int b_map;                                    // B loader lanes: 0 along k (k contiguous or nothing is), 1 along 8 rows x 4 k (rows contiguous)
  int MR, NB, KC;                               // full extents (rows of A, rows of B, contraction length)
  int n_tiles;                                  // 64-column tiles (gridDim.y = m_tiles * n_tiles)
  int KCp, kshift;                              // B loader mapping: min(KC, 32) rounded up to a power of two (>= 8)
  int conjA, a_early, b_early;                  // *_early: the operand is not written by the previous kernel of the stream
  int l2_prefetch;                              // 1: issue L2 prefetches ahead of the loads (operands expected in DRAM).  Off inside the
                                                // dense chains: their operands are L2-resident (fresh, or pulled in by the analysis
                                                // launch), and every prefetch costs an L1 wavefront per 32-byte sector like a load
  // fused bias gradient (dweight launch): dbias[o] = bias_scale * sum_b Re gm[b, o, dc]
  const float2* bias_gm; float* dbias; int bias_B, bias_Co, dc_quad; long long bias_sB, bias_sO; float bias_scale;   // bias_gm points at (b=0, o=0, DC)
  long long* trace;        // debug timeline of CTA 0 (SC_TRACE_FILE, -DSC_TRACE_QUAD builds only), else nullptr
};

__global__ void __launch_bounds__(MQ2_THREADS, 1) k_mode_gemm_quad2(const ModeGemmQuad2Params P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ uint64_t bar_a_full[MQ2_A_SLOTS], bar_a_empty[MQ2_A_SLOTS], bar_b_full[MQ2_B_SLOTS], bar_b_empty[MQ2_B_SLOTS], bar_d_full;
  __shared__ uint32_t tmem_base_slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int mt = (int)blockIdx.y / P.n_tiles, nt = (int)blockIdx.y % P.n_tiles;
  const int MR = min(64, P.MR - 64 * mt), NB = min(64, P.NB - 64 * nt);
  const int NBp = (NB + 15) & ~15;
  const int KC = P.KC;
  const int n_chunks = (KC + 7) >> 3, n_slabs = (KC + 31) >> 5;
  const long long qd = (long long)blockIdx.x;          // this CTA's quad of modes
  if (tid == 128) SC_QTRACE(P, 0, 0, 0);

  if (tid == 0) {
    for (int i = 0; i < MQ2_A_SLOTS; ++i) { mbar_init(&bar_a_full[i], MQ2_A_WARPS); mbar_init(&bar_a_empty[i], 1); }
    for (int i = 0; i < MQ2_B_SLOTS; ++i) { mbar_init(&bar_b_full[i], MQ2_B_WARPS); mbar_init(&bar_b_empty[i], 1); }
    mbar_init(&bar_d_full, 1);
    mbar_init_fence();
  }
  if (warp == 0) tmem_alloc(&tmem_base_slot, 512);
  if (NB < NBp || (KC & 7)) {   // padding rows / the K tail of B must hold finite values (zeros)
    uint4* z = reinterpret_cast<uint4*>(smem);
    const int n16 = (int)((n_slabs < MQ2_B_SLOTS ? n_slabs : MQ2_B_SLOTS) * (MQ2_SLAB_BYTES / 16));
    for (int i = tid; i < n16; i += MQ2_THREADS) z[i] = make_uint4(0, 0, 0, 0);
  }
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = tmem_base_slot;
  if (tid == 128) SC_QTRACE(P, 0, 0, 1);

  if (warp >= 4 + MQ2_A_WARPS) {
    // ------------------------------------------------------------------ B loaders: global -> registers -> bf16 hi / lo -> swizzled smem
    const int lt = tid - (4 + MQ2_A_WARPS) * 32;
    // lanes along k (32 consecutive k of one row: coalesced when k is the contiguous index) or 8 rows x 4 k per warp
    // (coalesced when the row is); either way a warp's swizzled stores touch 32 distinct banks
    const int kq = P.b_map ? (((lt >> 5) << 2) | ((lt >> 3) & 3)) : (lt & (P.KCp - 1));   // k within the 32-complex slab
    const int r0 = P.b_map ? (lt & 7) : (lt >> P.kshift);
    const int step = P.b_map ? 8 : ((MQ2_B_WARPS * 32) >> P.kshift);    // 8, 16 or 32 rows between a thread's elements
    const uint32_t off_hi = (uint32_t)(r0 * 128 + ((((2 * kq) >> 3) ^ r0) & 7) * 16 + ((2 * kq) & 7) * 2);
    const uint32_t off_lo = off_hi + (uint32_t)NBp * 128u;
    const uint32_t sstep = (uint32_t)step * 128u;
    const float2* base = P.b + qd * P.sBQ + (long long)(64 * nt + r0) * P.sBN;
    if (!P.b_early) pdl_wait();
    for (int rd = 0; rd < n_slabs; ++rd) {
      const int slot = rd % MQ2_B_SLOTS;
      if (lt < 32) SC_QTRACE(P, 1, rd, 0);
      const int k = rd * 32 + kq;
      const bool k_in = kq < 32 && k < ((KC + 7) & ~7);    // inside the K range the MMAs read
      const bool k_ok = k_in && k < KC;                    // real data (else: explicit zeros)
      const float2* pk = base + (long long)k * P.sBK;
      uint8_t* tile = smem + (size_t)slot * MQ2_SLAB_BYTES;
#pragma unroll
      for (int bt = 0; bt < 2; ++bt) {
        float v[4][8];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (k_ok && r0 + (4 * bt + u) * step < NB) ld_global_v8(pk + (long long)(4 * bt + u) * step * P.sBN, v[u]);
          else {
#pragma unroll
            for (int e = 0; e < 8; ++e) v[u][e] = 0.f;
          }
        }
        if (bt == 0) {
          if (P.l2_prefetch) {
#pragma unroll
            for (int u = 4; u < 8; ++u)
              if (k_ok && r0 + u * step < NB) prefetch_l2(pk + (long long)u * step * P.sBN);
            if (rd + 1 < n_slabs && kq < 32 && k + 32 < KC) {
#pragma unroll
              for (int u = 0; u < 8; ++u)
                if (r0 + u * step < NB) prefetch_l2(pk + 32 * P.sBK + (long long)u * step * P.sBN);
            }
          }
          if (rd >= MQ2_B_SLOTS) mbar_wait(&bar_b_empty[slot], (uint32_t)(((rd / MQ2_B_SLOTS) - 1) & 1));
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (k_in && r0 + (4 * bt + u) * step < NB) {
            uint8_t* t0 = tile + off_hi + (4 * bt + u) * sstep;
            uint8_t* t1 = tile + off_lo + (4 * bt + u) * sstep;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint32_t hi, lo;
              split2_bf16(v[u][2 * j], v[u][2 * j + 1], hi, lo);
              *reinterpret_cast<uint32_t*>(t0 + j * MQ2_MODE_BYTES) = hi;
              *reinterpret_cast<uint32_t*>(t1 + j * MQ2_MODE_BYTES) = lo;
            }
          }
        }
        if (lt < 32) SC_QTRACE(P, 1, rd, 1 + bt);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_b_full[slot]);
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ A loaders: global -> registers -> bf16 hi / lo -> tensor memory
    // thread <-> real row (lane of the TMEM quarter) and 4 of the 8 k of every chunk; the two lanes of a complex row read the
    // same sectors (one request after coalescing) and keep different arrangements of them
    const int aw = warp - 4, q = aw & 3, g = aw >> 2;
    const int row = 32 * q + lane, R = row >> 1, part = row & 1;
    const bool r_ok = R < MR;
    const float2* pa = P.a + qd * P.sAQ + (long long)(64 * mt + R) * P.sAR + (long long)(4 * g) * P.sAK;
    const uint32_t tm_mine = tmem + MQ2_TM_A + ((uint32_t)(32 * q) << 16) + (uint32_t)(4 * g);
    // sign / order of the packed (first K element | second K element << 16) pair for this row
    //   part 0: (re, -im)   conj: (re, im)        part 1: (im, re)   conj: (-im, re)
    const uint32_t flip = part == 0 ? (P.conjA ? 0u : 0x80000000u) : (P.conjA ? 0x00008000u : 0u);
    const uint32_t perm = part == 0 ? 0x3210u : 0x1032u;
    if (!P.a_early) pdl_wait();
    if (aw == 0) SC_QTRACE(P, 0, 0, 2);
    float v0[4][8], v1[4][8];
    auto issue = [&](float (&buf)[4][8], int c) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (r_ok && 8 * c + 4 * g + u < KC) ld_global_v8(pa + (long long)(8 * c + u) * P.sAK, buf[u]);
        else {
#pragma unroll
          for (int e = 0; e < 8; ++e) buf[u][e] = 0.f;
        }
      }
    };
    auto consume = [&](float (&buf)[4][8], int c) {
      const int s = c % MQ2_A_SLOTS;
      if (aw == 0) SC_QTRACE(P, 0, 1 + c, 0);
      if (c >= MQ2_A_SLOTS) {
        mbar_wait(&bar_a_empty[s], (uint32_t)(((c / MQ2_A_SLOTS) - 1) & 1));
        tc_fence_after_sync();
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t hw[4], lw[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          uint32_t hi, lo;
          split2_bf16(buf[u][2 * j], buf[u][2 * j + 1], hi, lo);      // (re | im << 16)
          hw[u] = __byte_perm(hi, 0, perm) ^ flip;
          lw[u] = __byte_perm(lo, 0, perm) ^ flip;
        }
        tmem_st4(tm_mine + (uint32_t)(64 * s + 16 * j), hw[0], hw[1], hw[2], hw[3]);
        tmem_st4(tm_mine + (uint32_t)(64 * s + 16 * j + 8), lw[0], lw[1], lw[2], lw[3]);
        if (j == 0 && aw == 0) SC_QTRACE(P, 0, 1 + c, 1);
      }
      tmem_st_wait();
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_a_full[s]);
      if (aw == 0) SC_QTRACE(P, 0, 1 + c, 2);
    };
    issue(v0, 0);
    if (n_chunks > 1) issue(v1, 1);
    if (r_ok && P.l2_prefetch) {
      for (int c = 2; c < n_chunks && c < 10; ++c)
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (8 * c + 4 * g + u < KC) prefetch_l2(pa + (long long)(8 * c + u) * P.sAK);
    }
    for (int c = 0; c < n_chunks; c += 2) {
      consume(v0, c);
      if (c + 2 < n_chunks) issue(v0, c + 2);
      if (c + 1 < n_chunks) {
        consume(v1, c + 1);
        if (c + 3 < n_chunks) issue(v1, c + 3);
      }
      if (r_ok && P.l2_prefetch && c + 10 < n_chunks) {
#pragma unroll
        for (int cc = c + 10; cc < c + 12; ++cc)
#pragma unroll
          for (int u = 0; u < 4; ++u)
            if (cc < n_chunks && 8 * cc + 4 * g + u < KC) prefetch_l2(pa + (long long)(8 * cc + u) * P.sAK);
      }
    }
  } else if (warp == 0) {
    // ------------------------------------------------------------------ MMA issue (one lane)
    if (lane == 0) {
      const uint32_t idesc = idesc_bf16(128, NBp);
      const uint32_t base_lo = desc_lo(smem_u32(smem));
      const uint32_t lo_rows = ((uint32_t)NBp * 128u) >> 4;
      for (int c = 0; c < n_chunks; ++c) {
        const int s = c % MQ2_A_SLOTS, slab = c >> 2, bslot = slab % MQ2_B_SLOTS;
        if ((c & 3) == 0) mbar_wait(&bar_b_full[bslot], (uint32_t)((slab / MQ2_B_SLOTS) & 1));
        mbar_wait(&bar_a_full[s], (uint32_t)((c / MQ2_A_SLOTS) & 1));
        tc_fence_after_sync();
        SC_QTRACE(P, 2, c, 0);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint32_t a_hi = tmem + MQ2_TM_A + (uint32_t)(64 * s + 16 * j), a_lo = a_hi + 8;
          const uint32_t b_hi = base_lo + (uint32_t)bslot * (MQ2_SLAB_BYTES >> 4) + (uint32_t)j * (MQ2_MODE_BYTES >> 4) + 2 * (uint32_t)(c & 3);
          const uint32_t d = tmem + (uint32_t)(64 * j);
          mma_bf16_ts(d, a_hi, desc_from_lo(b_hi), idesc, c > 0);
          mma_bf16_ts(d, a_hi, desc_from_lo(b_hi + lo_rows), idesc, true);
          mma_bf16_ts(d, a_lo, desc_from_lo(b_hi), idesc, true);
        }
        mma_commit(&bar_a_empty[s]);
        if ((c & 3) == 3 || c == n_chunks - 1) mma_commit(&bar_b_empty[bslot]);
        SC_QTRACE(P, 2, c, 1);
      }
      mma_commit(&bar_d_full);
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------------ dependency hand-over: the next kernel of the stream may
    // start once every CTA of this grid has seen its predecessor complete, so a kernel may read, ahead of its own wait, whatever
    // its immediate predecessor does not write
    pdl_wait();
    pdl_launch_dependents();
  }
  if (warp >= 1 && warp < 4 && P.dbias != nullptr && blockIdx.y == 0 && (int)blockIdx.x == P.dc_quad) {
    // fused bias gradient: dbias[o] = sum_b Re gm[b, o, DC] / synthesis scale (the DC slot of gm is the plain sum of gy)
    pdl_wait();
    for (int o = warp - 1; o < P.bias_Co; o += 3) {
      float sum = 0.f;
      for (int bb = lane; bb < P.bias_B; bb += 32) sum += __ldg(&P.bias_gm[(long long)bb * P.bias_sB + (long long)o * P.bias_sO].x);
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
      if (lane == 0) P.dbias[o] = sum * P.bias_scale;
    }
  }
  __syncwarp();
  {
    // ------------------------------------------------------------------ epilogue, ALL warps: four modes -> one 32-byte store
    const int q = warp & 3, grp = warp >> 2;
    const int row = q * 32 + lane;
    const int R = row >> 1, part = row & 1;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    pdl_wait();                                        // the output buffer may still be read by the previous kernel
    if (warp == 2) SC_QTRACE(P, 3, 0, 0);
    mbar_wait(&bar_d_full, 0);
    tc_fence_after_sync();
    if (warp == 2) SC_QTRACE(P, 3, 0, 1);
    float2* dst = P.out + qd * P.sOQ + (long long)(64 * mt + R) * P.sOR + (long long)(64 * nt) * P.sON;
    for (int c = 8 * grp; c < NBp; c += 8 * (MQ2_THREADS / 128)) {
      float acc[4][8];
#pragma unroll
      for (int j = 0; j < 4; ++j) tmem_ld8(tmem + lane_sel + (uint32_t)(j * 64 + c), acc[j]);
      tmem_ld_wait();
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float o[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float mine = acc[j][e];
          const float other = __shfl_xor_sync(0xffffffffu, mine, 1);
          o[2 * j] = mine; o[2 * j + 1] = other;      // (re, im) on even lanes
        }
        const int n = c + e;
        if (part == 0 && R < MR && n < NB) st_global_v8(reinterpret_cast<float*>(dst + (long long)n * P.sON), o);
      }
    }
    tc_fence_before_sync();
    if (warp == 2) SC_QTRACE(P, 3, 0, 2);
  }
  __syncthreads();
  if (warp == 2) SC_QTRACE(P, 3, 1, 0);
  if (warp == 0) tmem_dealloc(tmem, 512);
}

// =====================================================================================================
// mode-wise complex GEMM, four consecutive modes per CTA, third generation ("quad3"): quad2 fed by the TMA engine
//
//   Measured on quad2 (B200, round 2): its 256-bit loads of scattered 32-byte sectors complete at ~13-20 B/clk per SM -- the
//   LSU tracks each sector as its own request and the kernel spends ~15 000 of its ~21 000 cycles waiting for them --, whereas
//   4-D tensor loads with a {8 floats, 1 quad, 64 rows, 8 k} box gather the same sectors at 28 B/clk per SM with every box in
//   flight at once, no registers and no issue slots (sc_probe_tma_gather).  So here one producer lane streams both operands
//   into raw fp32 rings in shared memory and the converter warps only move shared memory -> registers -> tensor memory (A) /
//   swizzled bf16 tiles (B).  Tensor-memory ring, MMA issue and epilogue are quad2's.  K <= 64 (B tiles resident).
//   warp 0 MMA issue (+TMEM), warp 1 TMA producer + dependency hand-over, warps 2-3 fused bias gradient,
//   warps 4-11 A converters, 12-19 B converters, all 20 warps epilogue.
// =====================================================================================================
constexpr int MQ3_MAX_A_RAW = 8, MQ3_MAX_B_RAW = 2;
constexpr uint32_t MQ3_A_RAW_BYTES = 8 * 64 * 32;      // one chunk: [8 k][64 rows][4 modes x (re, im)]

struct ModeGemmQuad3Params {
  float2* out;
  long long sOR, sON, sOQ;                      // complex-element strides of the output (row, column, quad)
  int MR, NB, KC;                               // full extents
  int n_tiles;                                  // 64-column tiles (gridDim.y = m_tiles * n_tiles)
  int conjA, a_early, b_early;
  int n_a_raw, n_b_raw, b_box_rows;             // ring depths; rows of one B box (<= 64)
  // How the operands reach shared memory (chosen on the host from the strides):
  //   0  sectors scattered in memory: 4-D box {8 floats, 1 quad, rows, k}, one 32-byte request per sector; raw block [k][rows][32 B]
  //   1  (B only) k is the contiguous index (quad-major xm / gm as the B operand of the forward / dxm products): 3-D box
  //      {256 floats = 32 k, rows, 1 quad}, one 1 KB request per row; raw block [row][k][32 B]
  //   2  the row is the contiguous index (quad-major operands of the dweight product): 3-D boxes {256 floats = 32 rows, k, 1 quad},
  //      one 1 KB request per k and row half; raw block [row half][k][32 rows][32 B]
  int a_variant, b_variant;
  uint32_t tile_b_bytes, off_a_raw, off_b_raw, b_raw_bytes;
  const float2* bias_gm; float* dbias; int bias_B, bias_Co, dc_quad; long long bias_sB, bias_sO; float bias_scale;
  long long* trace;
};

__global__ void __launch_bounds__(MQ2_THREADS, 1) k_mode_gemm_quad3(const ModeGemmQuad3Params P, const __grid_constant__ CUtensorMap a_map,
                                                                      const __grid_constant__ CUtensorMap b_map) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ uint64_t bar_a_full[MQ2_A_SLOTS], bar_a_empty[MQ2_A_SLOTS], bar_b_full[2], bar_d_full;
  __shared__ uint64_t bar_ar_full[MQ3_MAX_A_RAW], bar_ar_empty[MQ3_MAX_A_RAW], bar_br_full[MQ3_MAX_B_RAW], bar_br_empty[MQ3_MAX_B_RAW];
  __shared__ uint32_t tmem_base_slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int mt = (int)blockIdx.y / P.n_tiles, nt = (int)blockIdx.y % P.n_tiles;
  const int MR = min(64, P.MR - 64 * mt), NB = min(64, P.NB - 64 * nt);
  const int NBp = (NB + 15) & ~15;
  const int KC = P.KC;
  const int n_chunks = (KC + 7) >> 3, n_slabs = (KC + 31) >> 5;
  const int qd = (int)blockIdx.x;
  const int NA = P.n_a_raw, NBR = P.n_b_raw;
  if (tid == 128) SC_QTRACE(P, 0, 0, 0);

  if (tid == 0) {
    for (int i = 0; i < MQ2_A_SLOTS; ++i) { mbar_init(&bar_a_full[i], MQ2_A_WARPS); mbar_init(&bar_a_empty[i], 1); }
    for (int i = 0; i < 2; ++i) mbar_init(&bar_b_full[i], MQ2_B_WARPS);
    for (int i = 0; i < NA; ++i) { mbar_init(&bar_ar_full[i], 1); mbar_init(&bar_ar_empty[i], MQ2_A_WARPS); }
    for (int i = 0; i < NBR; ++i) { mbar_init(&bar_br_full[i], 1); mbar_init(&bar_br_empty[i], MQ2_B_WARPS); }
    mbar_init(&bar_d_full, 1);
    mbar_init_fence();
  }
  if (warp == 0) tmem_alloc(&tmem_base_slot, 512);
  if (NB < NBp) {   // padding rows of the B tiles must hold finite values (zeros)
    uint4* z = reinterpret_cast<uint4*>(smem);
    const int n16 = (int)((uint32_t)(n_slabs * 4) * P.tile_b_bytes / 16);
    for (int i = tid; i < n16; i += MQ2_THREADS) z[i] = make_uint4(0, 0, 0, 0);
  }
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = tmem_base_slot;
  if (tid == 128) SC_QTRACE(P, 0, 0, 1);

  if (warp == 1) {
    // ------------------------------------------------------------------ TMA producer (one lane) + dependency hand-over
    if (lane == 0) {
      uint8_t* a_raw = smem + P.off_a_raw;
      uint8_t* b_raw = smem + P.off_b_raw;
      int ia = 0, ib = 0;
      auto issue_a = [&](int c) {
        const int slot = c % NA;
        if (c >= NA) mbar_wait(&bar_ar_empty[slot], (uint32_t)(((c / NA) - 1) & 1));
        mbar_arrive_expect_tx(&bar_ar_full[slot], MQ3_A_RAW_BYTES);
        tma_load_4d(a_raw + (size_t)slot * MQ3_A_RAW_BYTES, &a_map, &bar_ar_full[slot], 0, qd, 64 * mt, 8 * c);
      };
      auto issue_b = [&](int s) {
        const int slot = s % NBR;
        if (s >= NBR) mbar_wait(&bar_br_empty[slot], (uint32_t)(((s / NBR) - 1) & 1));
        mbar_arrive_expect_tx(&bar_br_full[slot], P.b_raw_bytes);
        tma_load_4d(b_raw + (size_t)slot * P.b_raw_bytes, &b_map, &bar_br_full[slot], 0, qd, 64 * nt, 32 * s);
      };
      // Consumption order: B slab s, then its A chunks 4s .. 4s+3.  Operands the previous kernel of the stream does not write
      // may be fetched ahead of the dependency wait -- at most two A chunks, so that they do not sit in the TMA queue in front of
      // the B slab the first MMA waits for.
      if (P.b_early) issue_b(ib++);
      if (P.a_early) while (ia < n_chunks && ia < 2) issue_a(ia++);
      pdl_wait();
      pdl_launch_dependents();   // (after the wait: see k_fused_analysis)
      SC_QTRACE(P, 0, 0, 2);
      while (ia < n_chunks || ib < n_slabs) {
        if (ib < n_slabs && 4 * ib <= ia) issue_b(ib++);
        else if (ia < n_chunks) issue_a(ia++);
        else issue_b(ib++);
      }
    }
    __syncwarp();
  } else if (warp >= 4 + MQ2_A_WARPS) {
    // ------------------------------------------------------------------ B converters: raw slab -> bf16 hi / lo -> swizzled tiles
    // a warp covers 8 rows x 4 k: 256 contiguous raw bytes per quarter-warp, 32 distinct banks on the swizzled side
    const int lt = tid - (4 + MQ2_A_WARPS) * 32;
    const int nlo = lt & 7, kq = ((lt >> 5) << 2) | ((lt >> 3) & 3);
    const uint32_t off_hi = (uint32_t)(nlo * 128 + ((((2 * kq) >> 3) ^ nlo) & 7) * 16 + ((2 * kq) & 7) * 2);
    const uint32_t off_lo = off_hi + (uint32_t)NBp * 128u;
    const int rows = P.b_box_rows;
    for (int s = 0; s < n_slabs; ++s) {
      const int slot = s % NBR;
      if (lt < 32) SC_QTRACE(P, 1, s, 0);
      mbar_wait(&bar_br_full[slot], (uint32_t)((s / NBR) & 1));
      if (lt < 32) SC_QTRACE(P, 1, s, 1);
      const uint8_t* src = smem + P.off_b_raw + (size_t)slot * P.b_raw_bytes + (size_t)(kq * rows + nlo) * 32;
      uint8_t* tile = smem + (size_t)(s * 4) * P.tile_b_bytes;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int n = nlo + 8 * u;
        if (n < NB) {
          const float4 lo4 = *reinterpret_cast<const float4*>(src + u * 256), hi4 = *reinterpret_cast<const float4*>(src + u * 256 + 16);
          const float v[8] = {lo4.x, lo4.y, lo4.z, lo4.w, hi4.x, hi4.y, hi4.z, hi4.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            uint32_t hi, lo;
            split2_bf16(v[2 * j], v[2 * j + 1], hi, lo);
            *reinterpret_cast<uint32_t*>(tile + j * P.tile_b_bytes + off_hi + u * 1024) = hi;
            *reinterpret_cast<uint32_t*>(tile + j * P.tile_b_bytes + off_lo + u * 1024) = lo;
          }
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) { mbar_arrive(&bar_br_empty[slot]); mbar_arrive(&bar_b_full[s]); }
      if (lt < 32) SC_QTRACE(P, 1, s, 2);
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ A converters: raw chunk -> bf16 hi / lo -> tensor memory
    const int aw = warp - 4, q = aw & 3, g = aw >> 2;
    const int row = 32 * q + lane, R = row >> 1, part = row & 1;
    const uint32_t tm_mine = tmem + MQ2_TM_A + ((uint32_t)(32 * q) << 16) + (uint32_t)(4 * g);
    //   part 0: (re, -im)   conj: (re, im)        part 1: (im, re)   conj: (-im, re)
    const uint32_t flip = part == 0 ? (P.conjA ? 0u : 0x80000000u) : (P.conjA ? 0x00008000u : 0u);
    const uint32_t perm = part == 0 ? 0x3210u : 0x1032u;
    const uint32_t my_raw = (uint32_t)((4 * g * 64 + R) * 32);
    for (int c = 0; c < n_chunks; ++c) {
      const int rs = c % NA, s = c % MQ2_A_SLOTS;
      if (aw == 0) SC_QTRACE(P, 0, 1 + c, 0);
      mbar_wait(&bar_ar_full[rs], (uint32_t)((c / NA) & 1));
      if (aw == 0) SC_QTRACE(P, 0, 1 + c, 1);
      const uint8_t* src = smem + P.off_a_raw + (size_t)rs * MQ3_A_RAW_BYTES + my_raw;
      uint32_t hw[4][4], lw[4][4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float4 lo4 = *reinterpret_cast<const float4*>(src + u * 2048), hi4 = *reinterpret_cast<const float4*>(src + u * 2048 + 16);
        const float v[8] = {lo4.x, lo4.y, lo4.z, lo4.w, hi4.x, hi4.y, hi4.z, hi4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t hi, lo;
          split2_bf16(v[2 * j], v[2 * j + 1], hi, lo);      // (re | im << 16)
          hw[j][u] = __byte_perm(hi, 0, perm) ^ flip;
          lw[j][u] = __byte_perm(lo, 0, perm) ^ flip;
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_ar_empty[rs]);       // the raw chunk has been consumed into registers
      if (c >= MQ2_A_SLOTS) {
        mbar_wait(&bar_a_empty[s], (uint32_t)(((c / MQ2_A_SLOTS) - 1) & 1));
        tc_fence_after_sync();
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        tmem_st4(tm_mine + (uint32_t)(64 * s + 16 * j), hw[j][0], hw[j][1], hw[j][2], hw[j][3]);
        tmem_st4(tm_mine + (uint32_t)(64 * s + 16 * j + 8), lw[j][0], lw[j][1], lw[j][2], lw[j][3]);
      }
      tmem_st_wait();
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_a_full[s]);
      if (aw == 0) SC_QTRACE(P, 0, 1 + c, 2);
    }
  } else if (warp == 0) {
    // ------------------------------------------------------------------ MMA issue (one lane)
    if (lane == 0) {
      const uint32_t idesc = idesc_bf16(128, NBp);
      const uint32_t base_lo = desc_lo(smem_u32(smem));
      const uint32_t lo_rows = ((uint32_t)NBp * 128u) >> 4;
      for (int c = 0; c < n_chunks; ++c) {
        const int s = c % MQ2_A_SLOTS, slab = c >> 2;
        if ((c & 3) == 0) mbar_wait(&bar_b_full[slab], 0);
        mbar_wait(&bar_a_full[s], (uint32_t)((c / MQ2_A_SLOTS) & 1));
        tc_fence_after_sync();
        SC_QTRACE(P, 2, c, 0);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint32_t a_hi = tmem + MQ2_TM_A + (uint32_t)(64 * s + 16 * j), a_lo = a_hi + 8;
          const uint32_t b_hi = base_lo + (uint32_t)(slab * 4 + j) * (P.tile_b_bytes >> 4) + 2 * (uint32_t)(c & 3);
          const uint32_t d = tmem + (uint32_t)(64 * j);
          mma_bf16_ts(d, a_hi, desc_from_lo(b_hi), idesc, c > 0);
          mma_bf16_ts(d, a_hi, desc_from_lo(b_hi + lo_rows), idesc, true);
          mma_bf16_ts(d, a_lo, desc_from_lo(b_hi), idesc, true);
        }
        mma_commit(&bar_a_empty[s]);
        SC_QTRACE(P, 2, c, 1);
      }
      mma_commit(&bar_d_full);
    }
    __syncwarp();
  } else if (P.dbias != nullptr && blockIdx.y == 0 && (int)blockIdx.x == P.dc_quad) {
    // ------------------------------------------------------------------ warps 2-3: fused bias gradient
    pdl_wait();
    for (int o = warp - 2; o < P.bias_Co; o += 2) {
      float sum = 0.f;
      for (int bb = lane; bb < P.bias_B; bb += 32) sum += __ldg(&P.bias_gm[(long long)bb * P.bias_sB + (long long)o * P.bias_sO].x);
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
      if (lane == 0) P.dbias[o] = sum * P.bias_scale;
    }
  }
  __syncwarp();
  {
    // ------------------------------------------------------------------ epilogue, ALL warps: four modes -> one 32-byte store
    const int q = warp & 3, grp = warp >> 2;
    const int row = q * 32 + lane;
    const int R = row >> 1, part = row & 1;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    pdl_wait();                                        // the output buffer may still be read by the previous kernel
    if (warp == 2) SC_QTRACE(P, 3, 0, 0);
    mbar_wait(&bar_d_full, 0);
    tc_fence_after_sync();
    if (warp == 2) SC_QTRACE(P, 3, 0, 1);
    float2* dst = P.out + (long long)qd * P.sOQ + (long long)(64 * mt + R) * P.sOR + (long long)(64 * nt) * P.sON;
    for (int c = 8 * grp; c < NBp; c += 8 * (MQ2_THREADS / 128)) {
      float acc[4][8];
#pragma unroll
      for (int j = 0; j < 4; ++j) tmem_ld8(tmem + lane_sel + (uint32_t)(j * 64 + c), acc[j]);
      tmem_ld_wait();
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float o[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float mine = acc[j][e];
          const float other = __shfl_xor_sync(0xffffffffu, mine, 1);
          o[2 * j] = mine; o[2 * j + 1] = other;      // (re, im) on even lanes
        }
        const int n = c + e;
        if (part == 0 && R < MR && n < NB) st_global_v8(reinterpret_cast<float*>(dst + (long long)n * P.sON), o);
      }
    }
    tc_fence_before_sync();
    if (warp == 2) SC_QTRACE(P, 3, 0, 2);
  }
  __syncthreads();
  if (warp == 2) SC_QTRACE(P, 3, 1, 0);
  if (warp == 0) tmem_dealloc(tmem, 512);
}

// The opt-in dynamic shared memory limit is a per-device property of a kernel: remember what was set per device ordinal.
constexpr int SC_MAX_DEVICES = 64;
struct SmemOptIn { std::atomic<uint32_t> bytes[SC_MAX_DEVICES]; };
static bool ensure_dynamic_smem(const void* kernel, SmemOptIn& set, int device, uint32_t bytes, const char* what) {
  const bool tracked = device >= 0 && device < SC_MAX_DEVICES;
  if (tracked && set.bytes[device].load(std::memory_order_relaxed) >= bytes) return true;
  if (!cuda_ok(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes), what)) return false;
  if (tracked) set.bytes[device].store(bytes, std::memory_order_relaxed);
  return true;
}

static int fast_sm_count(const Plan* p);   // defined with FastTables below
static long long* trace_begin();
static void trace_end(long long* d, const char* what);
static cudaError_t launch_pdl(const void* func, dim3 grid, dim3 block, size_t smem, cudaStream_t st, void** args);

static bool mode_gemm_tc_supported(int MR, int NB, int KC) {
  return MR >= 1 && MR <= 64 && NB >= 1 && NB <= 64 && KC >= 1 && KC <= 64;
}

static inline bool aligned32(const void* ptr) { return (reinterpret_cast<uintptr_t>(ptr) & 31u) == 0; }

static bool launch_mode_gemm_quad2(const Plan* p, const float2* a, long long sAR, long long sAK, bool conjA, const float2* b,
                                   long long sBN, long long sBK, float2* out, long long sOR, long long sON, int MR, int NB,
                                   int KC, int64_t n_modes, const ModeGemmExtras* ex, cudaStream_t st) {
  ModeGemmQuad2Params P{};
  P.a = a; P.b = b; P.out = out;
  P.sAR = sAR; P.sAK = sAK; P.sBN = sBN; P.sBK = sBK; P.sOR = sOR; P.sON = sON;
  P.MR = MR; P.NB = NB; P.KC = KC;
  const int m_tiles = (MR + 63) / 64;
  P.n_tiles = (NB + 63) / 64;
  P.KCp = 8; P.kshift = 3;
  const int kc_round = KC < 32 ? KC : 32;
  while (P.KCp < kc_round) { P.KCp *= 2; ++P.kshift; }
  P.conjA = conjA ? 1 : 0;
  P.sAQ = P.sBQ = P.sOQ = 4;
  P.l2_prefetch = 1;
  if (ex != nullptr) {
    P.a_early = ex->a_early ? 1 : 0; P.b_early = ex->b_early ? 1 : 0;
    P.l2_prefetch = ex->l2_resident ? 0 : 1;
    if (ex->sAQ) P.sAQ = ex->sAQ;
    if (ex->sBQ) P.sBQ = ex->sBQ;
    if (ex->sOQ) P.sOQ = ex->sOQ;
    if (ex->dbias != nullptr) {
      // gm is the B operand of the dweight product: rows n = o, k = b
      P.bias_gm = b + (long long)(p->dc_slot >> 2) * P.sBQ + (p->dc_slot & 3);
      P.bias_sB = sBK; P.bias_sO = sBN;
      P.dbias = ex->dbias; P.bias_B = KC; P.bias_Co = NB; P.dc_quad = p->dc_slot >> 2; P.bias_scale = ex->bias_scale;
    }
  }
  P.b_map = (sBN < sBK) ? 1 : 0;
  const uint32_t smem_bytes = MQ2_B_SLOTS * MQ2_SLAB_BYTES + 1024u;
  static SmemOptIn opt_in;
  if (!ensure_dynamic_smem((const void*)k_mode_gemm_quad2, opt_in, p->device, smem_bytes, "cudaFuncSetAttribute(k_mode_gemm_quad2)"))
    return false;
  count_launch();
#ifdef SC_TRACE_QUAD
  P.trace = trace_begin();
#endif
  void* args[] = {(void*)&P};
  const bool ok = cuda_ok(launch_pdl((const void*)k_mode_gemm_quad2, dim3((unsigned)(n_modes / 4), (unsigned)(m_tiles * P.n_tiles)),
                                     dim3(MQ2_THREADS), smem_bytes, st, args),
                          "k_mode_gemm_quad2 launch");
#ifdef SC_TRACE_QUAD
  trace_end(P.trace, conjA ? (sBN < sBK ? "quad2 dweight" : "quad2 dxm") : "quad2 fwd");
#endif
  return ok;
}

static bool make_sector_gather_map(CUtensorMap* map, const float2* base, uint64_t n_quads, uint64_t n_rows, uint64_t n_k,
                                   uint64_t stride_quad_bytes, uint64_t stride_row_bytes, uint64_t stride_k_bytes, uint32_t box_rows,
                                   uint32_t box_k);

static bool cached_gather_map(const Plan* p, const float2* base, uint64_t nq, uint64_t rows, uint64_t k, uint64_t sq, uint64_t sr,
                              uint64_t sk, uint32_t box_rows, uint32_t box_k, CUtensorMap* out);

static bool cached_wide_map(const Plan* p, const float2* base, uint64_t inner_floats, uint64_t n_second, uint64_t nq, uint64_t stride_second_bytes,
                            uint64_t stride_quad_bytes, uint32_t box_inner, uint32_t box_second, CUtensorMap* out, uint32_t box_quads = 1);
// SC_WIDE_BOXES=0: every operand through the 32-byte-sector gather boxes (A/B runs)
static bool wide_boxes_enabled() { return false; }   // (the converters of this build read the sector-gather layout only)
// SC_QUAD3=0 keeps the LSU-fed quad2 kernel (A/B runs)
static bool quad3_enabled() {
  static const bool v = [] { const char* e = getenv("SC_QUAD3"); return e == nullptr || atoi(e) != 0; }();
  return v;
}

// returns false with *handled = false when the shape does not fit the TMA-fed kernel (the caller then runs quad2)
static bool launch_mode_gemm_quad3(const Plan* p, const float2* a, long long sAR, long long sAK, bool conjA, const float2* b,
                                   long long sBN, long long sBK, float2* out, long long sOR, long long sON, int MR, int NB,
                                   int KC, int64_t n_modes, const ModeGemmExtras* ex, cudaStream_t st, bool* handled) {
  *handled = false;
  if (!quad3_enabled() || KC > 64) return true;
  const long long sAQ = ex != nullptr && ex->sAQ ? ex->sAQ : 4, sBQ = ex != nullptr && ex->sBQ ? ex->sBQ : 4, sOQ = ex != nullptr && ex->sOQ ? ex->sOQ : 4;
  // tensor-map strides are byte counts that must be multiples of 16 and below 2^40
  const long long strides[6] = {sAQ, sAR, sAK, sBQ, sBN, sBK};
  for (long long v : strides) if (v <= 0 || (v & 1) != 0 || v * 8 >= (1ll << 40)) return true;
  ModeGemmQuad3Params P{};
  P.out = out; P.sOR = sOR; P.sON = sON; P.sOQ = sOQ;
  P.MR = MR; P.NB = NB; P.KC = KC;
  const int m_tiles = (MR + 63) / 64;
  P.n_tiles = (NB + 63) / 64;
  P.conjA = conjA ? 1 : 0;
  const int n_chunks = (KC + 7) / 8, n_slabs = (KC + 31) / 32;
  const int nb_max = NB < 64 ? NB : 64;
  P.b_box_rows = nb_max;
  const uint32_t nbp_max = (uint32_t)((nb_max + 15) / 16 * 16);
  P.tile_b_bytes = 2u * nbp_max * 128u;
  P.a_variant = (sAR == 4 && wide_boxes_enabled()) ? 2 : 0;
  P.b_variant = !wide_boxes_enabled() ? 0 : (sBK == 4 ? 1 : (sBN == 4 ? 2 : 0));
  P.b_raw_bytes = 32u * (uint32_t)nb_max * 32u;      // one raw K-slab: [32 k][nb_max rows][32 B] = nb_max KB
  if (P.b_variant == 2 && nb_max > 32) P.b_raw_bytes = 65536u;   // two full 32-row boxes (rows past NB are zero-filled)
  const uint32_t budget = 227u * 1024u - 2048u;
  const uint32_t b_tiles = (uint32_t)(n_slabs * 4) * P.tile_b_bytes;
  P.n_b_raw = n_slabs < 2 ? n_slabs : 2;
  if (b_tiles + (uint32_t)P.n_b_raw * P.b_raw_bytes + 2u * MQ3_A_RAW_BYTES > budget) P.n_b_raw = 1;
  if (b_tiles + (uint32_t)P.n_b_raw * P.b_raw_bytes + 2u * MQ3_A_RAW_BYTES > budget) return true;
  P.off_b_raw = (b_tiles + 1023u) & ~1023u;
  P.off_a_raw = P.off_b_raw + (uint32_t)P.n_b_raw * P.b_raw_bytes;
  int na = (int)((budget - P.off_a_raw) / MQ3_A_RAW_BYTES);
  if (na > n_chunks) na = n_chunks;
  if (na > MQ3_MAX_A_RAW) na = MQ3_MAX_A_RAW;
  if (na < 2 && n_chunks > 1) return true;
  P.n_a_raw = na;
  const uint32_t smem_bytes = P.off_a_raw + (uint32_t)na * MQ3_A_RAW_BYTES + 1024u;
  if (ex != nullptr) {
    P.a_early = ex->a_early ? 1 : 0; P.b_early = ex->b_early ? 1 : 0;
    if (ex->dbias != nullptr) {
      P.bias_gm = b + (long long)(p->dc_slot >> 2) * sBQ + (p->dc_slot & 3);
      P.bias_sB = sBK; P.bias_sO = sBN;
      P.dbias = ex->dbias; P.bias_B = KC; P.bias_Co = NB; P.dc_quad = p->dc_slot >> 2; P.bias_scale = ex->bias_scale;
    }
  }
  CUtensorMap a_map, b_map;
  const uint64_t nq = (uint64_t)(n_modes / 4);
  if (P.a_variant == 2) {   // rows contiguous: {8 * MR floats, KC, quads}, box {256 floats = 32 rows, 8 k, 1}
    if (!cached_wide_map(p, a, (uint64_t)MR * 8, (uint64_t)KC, nq, (uint64_t)sAK * 8, (uint64_t)sAQ * 8, 256, 8, &a_map)) return false;
  } else if (!cached_gather_map(p, a, nq, (uint64_t)MR, (uint64_t)KC, (uint64_t)sAQ * 8, (uint64_t)sAR * 8, (uint64_t)sAK * 8, 64, 8, &a_map)) {
    return false;
  }
  if (P.b_variant == 1) {          // k contiguous: {8 * KC floats, NB rows, quads}, box {256 floats = 32 k, rows, 1}
    if (!cached_wide_map(p, b, (uint64_t)KC * 8, (uint64_t)NB, nq, (uint64_t)sBN * 8, (uint64_t)sBQ * 8, 256, (uint32_t)nb_max, &b_map)) return false;
  } else if (P.b_variant == 2) {   // rows contiguous: {8 * NB floats, KC, quads}, box {256 floats = 32 rows, 32 k, 1}
    if (!cached_wide_map(p, b, (uint64_t)NB * 8, (uint64_t)KC, nq, (uint64_t)sBK * 8, (uint64_t)sBQ * 8, (uint32_t)(nb_max < 32 ? nb_max * 8 : 256), 32,
                         &b_map))
      return false;
  } else if (!cached_gather_map(p, b, nq, (uint64_t)NB, (uint64_t)KC, (uint64_t)sBQ * 8, (uint64_t)sBN * 8, (uint64_t)sBK * 8, (uint32_t)nb_max, 32,
                                &b_map)) {
    return false;
  }
  static SmemOptIn opt_in;
  if (!ensure_dynamic_smem((const void*)k_mode_gemm_quad3, opt_in, p->device, smem_bytes, "cudaFuncSetAttribute(k_mode_gemm_quad3)"))
    return false;
  count_launch();
#ifdef SC_TRACE_QUAD
  P.trace = trace_begin();
#endif
  void* args[] = {(void*)&P, (void*)&a_map, (void*)&b_map};
  const bool ok = cuda_ok(launch_pdl((const void*)k_mode_gemm_quad3, dim3((unsigned)(n_modes / 4), (unsigned)(m_tiles * P.n_tiles)),
                                     dim3(MQ2_THREADS), smem_bytes, st, args),
                          "k_mode_gemm_quad3 launch");
#ifdef SC_TRACE_QUAD
  trace_end(P.trace, conjA ? (sBN < sBK ? "quad3 dweight" : "quad3 dxm") : "quad3 fwd");
#endif
  *handled = ok;
  return ok;
}

bool quad2_enabled() { return true; }

bool mode_gemm_quad_eligible(const Plan* p, int64_t n_modes, const void* a, const void* b, const void* out) {
  return p->fast != nullptr && p->weight_block_is_whole && n_modes % 4 == 0 && aligned32(a) && aligned32(b) && aligned32(out);
}

bool launch_mode_gemm_tc(const Plan* p, const float2* a, long long sAR, long long sAK, const int* offA, bool conjA,
                         const float2* b, long long sBN, long long sBK, const int* offB, float2* out, long long sOR,
                         long long sON, const int* offO, int MR, int NB, int KC, int64_t n_modes, cudaStream_t st,
                         ModeGemmExtras* ex) {
  // Quad variants: modes contiguous in every operand (no sliced weight block), every stride a multiple of 4 complex
  // elements and 32-byte aligned bases, so that 4 consecutive modes are exactly one sector.
  const bool contiguous = (offA == nullptr || p->weight_block_is_whole) && (offB == nullptr || p->weight_block_is_whole) &&
                          (offO == nullptr || p->weight_block_is_whole);
  const bool strides4 = ((sAR | sAK | sBN | sBK | sOR | sON) & 3) == 0;
  if (contiguous && strides4 && n_modes % 4 == 0 && aligned32(a) && aligned32(b) && aligned32(out)) {
    bool handled = false;
    if (!launch_mode_gemm_quad3(p, a, sAR, sAK, conjA, b, sBN, sBK, out, sOR, sON, MR, NB, KC, n_modes, ex, st, &handled)) return false;
    if (!handled && !launch_mode_gemm_quad2(p, a, sAR, sAK, conjA, b, sBN, sBK, out, sOR, sON, MR, NB, KC, n_modes, ex, st)) return false;
    if (ex != nullptr && ex->dbias != nullptr) ex->bias_done = true;
    return true;
  }
  if (!mode_gemm_tc_supported(MR, NB, KC)) { set_error("launch_mode_gemm_tc: extents above 64 need the quad layout"); return false; }
  ModeGemmTcParams P{};
  P.a = a; P.b = b; P.out = out;
  P.sAR = sAR; P.sAK = sAK; P.sBN = sBN; P.sBK = sBK; P.sOR = sOR; P.sON = sON;
  P.offA = offA; P.offB = offB; P.offO = offO;
  P.MR = MR; P.NB = NB; P.KC = KC;
  P.NBp = (NB + 15) / 16 * 16;   // N of an M=128 MMA must be a multiple of 16
  P.Kreal = (2 * KC + 63) / 64 * 64;
  P.KCp = 8; P.kshift = 3;
  while (P.KCp < KC) { P.KCp *= 2; ++P.kshift; }
  P.conjA = conjA ? 1 : 0;
  P.n_modes = (int)n_modes;
  const uint32_t a_bytes = 128u * (uint32_t)P.Kreal * 2u;
  const uint32_t b_bytes = 2u * (uint32_t)P.NBp * (uint32_t)P.Kreal * 2u;
  P.off_alo = a_bytes;
  P.off_b = 2 * a_bytes;
  P.stage_bytes = (2 * a_bytes + b_bytes + 1023u) & ~1023u;
  const uint32_t smem_bytes = 2 * P.stage_bytes + 1024u;
  static SmemOptIn opt_in;
  if (!ensure_dynamic_smem((const void*)k_mode_gemm_tc, opt_in, p->device, smem_bytes, "cudaFuncSetAttribute(k_mode_gemm_tc)"))
    return false;
  const int sms = fast_sm_count(p);
  // contiguous mode ranges, a multiple of 4 modes (one 32-byte sector of complex64) per CTA
  int per = (int)((n_modes + sms - 1) / sms);
  per = (per + 3) / 4 * 4;
  P.modes_per_cta = per;
  const int grid = (int)((n_modes + per - 1) / per);
  k_mode_gemm_tc<<<grid, MG2_THREADS, smem_bytes, st>>>(P);
  count_launch();
  return cuda_ok(cudaGetLastError(), "k_mode_gemm_tc launch");
}

// quad_ok: the operands qualify for the quad kernels (mode_gemm_quad_eligible), which take any extents; the single-mode
// tensor-core kernel (sliced weight blocks, unaligned bases) is limited to 64 x 64 x 64
bool fast_can_contract(const Plan* p, int B, int Ci, int Co, bool quad_ok) {
  if (p->fast == nullptr) return false;
  if (quad_ok) return true;
  return mode_gemm_tc_supported(Co, B, Ci) && mode_gemm_tc_supported(Ci, B, Co) && mode_gemm_tc_supported(Ci, Co, B);
}

// ---------------------------------------------------------------------------------------------------------
// host side: operand images and dispatch
// ---------------------------------------------------------------------------------------------------------
struct FusedAnalysisTables {
  bool ok = false;
  bool v2_ok = false;       // k_fused_analysis2 (x operand in tensor memory) applies
  int v2_stages = 0;
  uint32_t v2_off_b1 = 0, v2_off_b2 = 0, v2_off_scratch = 0, v2_smem_bytes = 0;
  int W = 0, H = 0, G = 0, N1 = 0, KX = 0, KY = 0, slabs = 0, n_stages = 0, tmem_cols = 0;
  uint8_t* d_b1 = nullptr;
  uint8_t* d_a2 = nullptr;
  uint32_t off_f32 = 0, off_ring = 0, off_b1 = 0, off_a2 = 0, off_b2 = 0, off_scratch = 0, stage_off = 0, smem_bytes = 0;
};

struct FusedSynthesisTables {
  bool ok = false;
  int W = 0, H = 0, G = 0, N1 = 0, KX = 0, KY = 0, tmem_cols = 0;
  uint8_t* d_aa = nullptr;
  uint8_t* d_bb = nullptr;
  uint32_t off_aa = 0, off_ba = 0, off_u = 0, off_bb = 0, off_stage = 0, smem_bytes = 0;
};

// Encoding a CUtensorMap costs tens of microseconds on the host; training loops hand the same buffers (PyTorch's caching
// allocator) to the same plan step after step, so encoded maps are kept in a small per-plan cache.
struct TensorMapCacheEntry { const void* base; uint64_t rows, W; int kind; CUtensorMap map; };

// last-dim ("rows") tensor-core kernels for grids the fused 2-D kernels do not cover -- see the section at the end of the file
struct RowsAnaTables {
  bool ok = false;
  int W = 0, N1 = 0, out_cols = 0, slabs = 0, f32_stages = 0, ring_stages = 0, tmem_cols = 0;
  uint32_t tab_bytes = 0, slot_bytes = 0, off_f32 = 0, off_ring = 0, smem_bytes = 0;
  uint8_t* d_tab = nullptr;
};
struct RowsSynTables {
  bool ok = false;
  int W = 0, N1 = 0, in_cols = 0, n_chunks = 0, tmem_cols = 0;
  uint32_t u_bytes = 0, chunk_bytes = 0, off_a = 0, off_ustage = 0, off_tab = 0, off_stage = 0, smem_bytes = 0;
  uint8_t* d_tab = nullptr;
};

struct GatherMapCacheEntry { const void* base; uint64_t nq, rows, k, sq, sr, sk; uint32_t box_rows, box_k; CUtensorMap map; };

struct FastTables {
  std::vector<GatherMapCacheEntry> gather_cache;
  std::vector<TensorMapCacheEntry> map_cache;
  std::mutex map_mutex;
  FusedAnalysisTables ana[2];   // [0] forward analysis on `grid`, [1] adjoint-of-synthesis analysis on `out_grid`
  FusedSynthesisTables syn[2];  // [0] forward synthesis onto `out_grid`, [1] adjoint-of-analysis synthesis onto `grid`
  RowsAnaTables rows_ana[2];    // same indexing as `ana`
  RowsSynTables rows_syn[2];    // same indexing as `syn`
  int sm_count = 0;
};

static int fast_sm_count(const Plan* p) { return p->fast->sm_count; }
// CTAs of a persistent transform launch: one per SM, minus the SMs reserved for a concurrent collective (sc_plan_set_reserved_sms)
static thread_local bool t_reserve_sms = false;   // set by sc_backward_dense around the launches a collective runs next to
void fast_set_reserve(bool on) { t_reserve_sms = on; }
static int persistent_grid(const Plan* p, int n_tiles) {
  int sms = p->fast->sm_count - (t_reserve_sms ? p->reserved_sms : 0);
  if (sms < 1) sms = 1;
  return n_tiles < sms ? n_tiles : sms;
}

static bool make_slab_load_map(CUtensorMap* map, const float* base, uint64_t rows, uint64_t W);
static bool make_row_tile_map(CUtensorMap* map, float* base, uint64_t rows, uint64_t W);
typedef CUresult (*CtxGetCurrentFn)(CUcontext*);
static bool thread_has_context() {
  static const CtxGetCurrentFn fn = [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuCtxGetCurrent", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      return reinterpret_cast<CtxGetCurrentFn>(ptr);
    return static_cast<CtxGetCurrentFn>(nullptr);
  }();
  if (fn == nullptr) return true;   // cannot tell: leave the runtime alone
  CUcontext ctx = nullptr;
  return fn(&ctx) != CUDA_SUCCESS || ctx != nullptr;
}

static bool make_swizzled_box_map(CUtensorMap* map, const float* base, uint64_t rows, uint64_t W);
static bool make_16bit_map(CUtensorMap* map, const void* base, uint64_t rows, uint64_t W, int storage, bool store);
// kind 0: x slab loads, kind 1: image row-tile stores, kind 2: x loads as 128-byte-swizzled [128 x 32] boxes (k_fused_analysis2),
// kinds 3 / 4: the 16-bit x loads / dx stores of make_16bit_map, with storage = SC_FLAG_GRID_F16 / SC_FLAG_GRID_BF16
static bool cached_map(const Plan* p, int kind, const void* base, uint64_t rows, uint64_t W, CUtensorMap* out, int storage = 0) {
  if (storage != 0) kind += 8 * storage;   // distinct cache keys per element type
  FastTables* f = p->fast;
  std::lock_guard<std::mutex> lock(f->map_mutex);
  for (const TensorMapCacheEntry& e : f->map_cache)
    if (e.base == base && e.rows == rows && e.W == W && e.kind == kind) { *out = e.map; return true; }
  // cuTensorMapEncodeTiled is a driver entry point: it needs the primary context bound to THIS thread.  PyTorch's autograd
  // worker threads only get one lazily (first runtime call that needs it), and a backward whose allocations are all served
  // from the caching allocator reaches this point before any such call -- cudaFree(0) binds it.  Only when the thread really
  // has no context: cudaFree is not allowed while a stream capture is in progress (graph capture reaches this point with
  // buffers from the graph's private pool, i.e. cache misses), and a capturing thread always has its context.
  if (!thread_has_context()) cudaFree(nullptr);
  TensorMapCacheEntry e{base, rows, W, kind, {}};
  const int base_kind = kind % 8;
  const bool ok = storage != 0 ? make_16bit_map(&e.map, base, rows, W, storage, base_kind == 4)
                  : kind == 0 ? make_slab_load_map(&e.map, static_cast<const float*>(base), rows, W)
                  : kind == 2 ? make_swizzled_box_map(&e.map, static_cast<const float*>(base), rows, W)
                              : make_row_tile_map(&e.map, static_cast<float*>(const_cast<void*>(base)), rows, W);
  if (!ok) return false;
  if (f->map_cache.size() >= 32) f->map_cache.erase(f->map_cache.begin());
  f->map_cache.push_back(e);
  *out = e.map;
  return true;
}

static bool cached_gather_map(const Plan* p, const float2* base, uint64_t nq, uint64_t rows, uint64_t k, uint64_t sq, uint64_t sr,
                              uint64_t sk, uint32_t box_rows, uint32_t box_k, CUtensorMap* out) {
  FastTables* f = p->fast;
  std::lock_guard<std::mutex> lock(f->map_mutex);
  for (const GatherMapCacheEntry& e : f->gather_cache)
    if (e.base == base && e.nq == nq && e.rows == rows && e.k == k && e.sq == sq && e.sr == sr && e.sk == sk && e.box_rows == box_rows &&
        e.box_k == box_k) { *out = e.map; return true; }
  if (!thread_has_context()) cudaFree(nullptr);   // (see cached_map)
  GatherMapCacheEntry e{base, nq, rows, k, sq, sr, sk, box_rows, box_k, {}};
  if (!make_sector_gather_map(&e.map, base, nq, rows, k, sq, sr, sk, box_rows, box_k)) return false;
  if (f->gather_cache.size() >= 48) f->gather_cache.erase(f->gather_cache.begin());
  f->gather_cache.push_back(e);
  *out = e.map;
  return true;
}

static inline uint16_t bf16_bits(float f) {   // round to nearest even
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
static inline float bf16_to_float(uint16_t b) {
  uint32_t u = (uint32_t)b << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}
static inline size_t host_sw128_offset(int r, int k, int rows) {
  const int slab = k >> 6, kk = k & 63;
  return (size_t)slab * rows * 128 + (size_t)r * 128 + ((((kk >> 3) ^ r) & 7) << 4) + ((kk & 7) << 1);
}
// writes v as T1 (row r1) and T2 (row r2) of a [rows x K] K-major SW128 bf16 image
static inline void put_split(std::vector<uint8_t>& img, int rows, int r1, int r2, int k, float v) {
  const uint16_t t1 = bf16_bits(v);
  const uint16_t t2 = bf16_bits(v - bf16_to_float(t1));
  memcpy(&img[host_sw128_offset(r1, k, rows)], &t1, 2);
  memcpy(&img[host_sw128_offset(r2, k, rows)], &t2, 2);
}

template <typename T>
static bool upload_bytes(Plan* p, const std::vector<T>& host, uint8_t** dev) {
  void* d = nullptr;
  if (!cuda_ok(cudaMalloc(&d, host.size() * sizeof(T)), "cudaMalloc(fast table)")) return false;
  p->owned.push_back(d);
  if (!cuda_ok(cudaMemcpy(d, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice), "cudaMemcpy(fast table)")) return false;
  *dev = static_cast<uint8_t*>(d);
  return true;
}

// last-dim table `tab` is [W x 2KX] (row stride 2KX); leading-dim table `lead` is [KY x H] complex
static bool build_fused_analysis(Plan* p, FusedAnalysisTables* t, int H, int W, int KY, int KX, const std::vector<float>& tab,
                                 const std::vector<float2>& lead) {
  t->ok = false;
  if (W % 64 != 0 || W > 128 || H < 16 || 128 % H != 0) return true;
  const int G = 128 / H;
  const int N1 = ((2 * KX + 15) / 16) * 16;
  if (N1 > 64 || G * KY > 32 || KX < 1 || KY < 1) return true;   // TMEM: D1[2] + D2[2] + the 128-column table = 6*N1 + 128 <= 512
  t->W = W; t->H = H; t->G = G; t->N1 = N1; t->KX = KX; t->KY = KY; t->slabs = W / 64;
  t->tmem_cols = 6 * N1 + 128 <= 256 ? 256 : 512;
  // ---- B1: [2*N1 x W]
  std::vector<uint8_t> b1((size_t)2 * N1 * W * 2, 0);
  for (int j = 0; j < 2 * KX; ++j)
    for (int w = 0; w < W; ++w) put_split(b1, 2 * N1, j, N1 + j, w, tab[(size_t)w * 2 * KX + j]);
  // ---- A2: [128 x 256]; row i' = 2*(g*KY + ky) + p_out (T1), 64 + i' (T2); column k2 = 2*(g*H + h) + p_in
  std::vector<uint16_t> a2((size_t)128 * 256, 0);   // plain row-major [row][k2]
  auto put_plain = [&](int r1, int r2, int k, float v) {
    const uint16_t t1 = bf16_bits(v);
    a2[(size_t)r1 * 256 + k] = t1;
    a2[(size_t)r2 * 256 + k] = bf16_bits(v - bf16_to_float(t1));
  };
  for (int g = 0; g < G; ++g)
    for (int ky = 0; ky < KY; ++ky)
      for (int h = 0; h < H; ++h) {
        const float2 f = lead[(size_t)ky * H + h];
        const int q = g * KY + ky, hl = g * H + h;
        put_plain(2 * q + 0, 64 + 2 * q + 0, 2 * hl + 0, f.x);
        put_plain(2 * q + 0, 64 + 2 * q + 0, 2 * hl + 1, -f.y);
        put_plain(2 * q + 1, 64 + 2 * q + 1, 2 * hl + 0, f.y);
        put_plain(2 * q + 1, 64 + 2 * q + 1, 2 * hl + 1, f.x);
      }
  if (!upload_bytes(p, b1, &t->d_b1) || !upload_bytes(p, a2, &t->d_a2)) return false;
  // ---- shared-memory carve-up
  if ((G * KY * KX) % 2 != 0) return true;   // the per-tile mode block is stored with one 16-byte-granular bulk copy
  const uint32_t scr_bytes = (64u * (uint32_t)(N1 / 2 + 1) * 4u + 15u) & ~15u;
  const uint32_t scratch_total = (scr_bytes + 2u * (uint32_t)(G * KY * KX) * 8u + 1023u) & ~1023u;
  t->stage_off = scr_bytes;
  const uint32_t fixed = (uint32_t)b1.size() + (uint32_t)N1 * 512u + scratch_total;   // B1 + B2 + scratch (the leading-dim table lives in TMEM)
  // [fp32 staging: FA_F32_STAGES slabs x 32 KB][bf16 hi/lo ring: `stages` x 32 KB][B1][B2][scratch]
  const uint32_t f32_bytes = (uint32_t)FA_F32_STAGES * 32768u;
  int stages = (int)(((227u * 1024u - 4096u - fixed) - f32_bytes) / FA_STAGE_BYTES);
  if (227u * 1024u - 4096u < fixed + f32_bytes + FA_STAGE_BYTES) return true;
  if (stages > 4) stages = 4;
  if (stages < 1) return true;
  t->n_stages = stages;
  t->off_f32 = 0;
  t->off_ring = f32_bytes;
  t->off_b1 = t->off_ring + (uint32_t)stages * FA_STAGE_BYTES;
  t->off_a2 = t->off_b1 + (uint32_t)b1.size();
  t->off_b2 = t->off_a2;
  t->off_scratch = t->off_b2 + (uint32_t)N1 * 512u;
  t->smem_bytes = t->off_scratch + scratch_total + 1024u;
  t->ok = true;
  // second generation: no bf16 operand ring; fp32 staging as deep as shared memory allows
  if (5 * N1 + 128 + 64 * FA2_X_STAGES <= 512) {
    int st2 = (int)((227u * 1024u - 4096u - fixed) / 32768u);
    if (st2 > FA2_MAX_F32) st2 = FA2_MAX_F32;
    if (st2 >= 2) {
      t->v2_ok = true;
      t->v2_stages = st2;
      t->v2_off_b1 = (uint32_t)st2 * 32768u;
      t->v2_off_b2 = t->v2_off_b1 + (uint32_t)b1.size();
      t->v2_off_scratch = t->v2_off_b2 + (uint32_t)N1 * 512u;
      t->v2_smem_bytes = t->v2_off_scratch + scratch_total + 1024u;
    }
  }
  return true;
}

// last-dim table `tab` is [2KX x W] (row stride W); leading-dim table `lead` is [H x KY] complex
static bool build_fused_synthesis(Plan* p, FusedSynthesisTables* t, int H, int W, int KY, int KX, const std::vector<float>& tab,
                                  const std::vector<float2>& lead) {
  t->ok = false;
  if (W % 64 != 0 || W > 256 || H < 16 || 128 % H != 0) return true;
  const int G = 128 / H;
  const int N1 = ((2 * KX + 15) / 16) * 16;
  if (N1 > 64 || G * KY > 32 || KX < 1 || KY < 1 || 4 * N1 + 2 * W > 512) return true;
  t->W = W; t->H = H; t->G = G; t->N1 = N1; t->KX = KX; t->KY = KY;
  t->tmem_cols = 4 * N1 + 2 * W <= 256 ? 256 : 512;
  // ---- AA: [128 x 128]; row hl = g*H + h; columns 2q+s (T1) and 64+2q+s (T2), q = g*KY + ky, s: 0 = Re, 1 = Im of the table
  std::vector<uint8_t> aa((size_t)128 * 128 * 2, 0);
  {
    // T1 and T2 of the same coefficient live in the SAME row at columns k and 64 + k
    for (int g = 0; g < G; ++g)
      for (int h = 0; h < H; ++h)
        for (int ky = 0; ky < KY; ++ky) {
          const float2 f = lead[(size_t)h * KY + ky];
          const int hl = g * H + h, q = g * KY + ky;
          const float vals[2] = {f.x, f.y};
          for (int sgn = 0; sgn < 2; ++sgn) {
            const uint16_t t1 = bf16_bits(vals[sgn]);
            const uint16_t t2 = bf16_bits(vals[sgn] - bf16_to_float(t1));
            memcpy(&aa[host_sw128_offset(hl, 2 * q + sgn, 128)], &t1, 2);
            memcpy(&aa[host_sw128_offset(hl, 64 + 2 * q + sgn, 128)], &t2, 2);
          }
        }
  }
  // ---- BB: T1 image then T2 image, each [W x 64]: row w, column j
  std::vector<uint8_t> bb((size_t)2 * W * 128, 0);
  for (int j = 0; j < 2 * KX; ++j)
    for (int w = 0; w < W; ++w) {
      const float v = tab[(size_t)j * W + w];
      const uint16_t t1 = bf16_bits(v);
      const uint16_t t2 = bf16_bits(v - bf16_to_float(t1));
      memcpy(&bb[host_sw128_offset(w, j, W)], &t1, 2);
      memcpy(&bb[(size_t)W * 128 + host_sw128_offset(w, j, W)], &t2, 2);
    }
  if (!upload_bytes(p, aa, &t->d_aa) || !upload_bytes(p, bb, &t->d_bb)) return false;
  t->off_aa = 0;
  t->off_ba = 32768u;
  t->off_u = t->off_ba + 2u * (uint32_t)(2 * N1 * 256);
  t->off_bb = t->off_u + 2u * (uint32_t)(2 * FA_SLAB_BYTES);
  t->off_stage = t->off_bb + (uint32_t)bb.size();
  t->off_stage = (t->off_stage + 1023u) & ~1023u;
  t->smem_bytes = t->off_stage + FS_STAGE_BYTES + 1024u;
  if (t->smem_bytes > 227u * 1024u - 4096u) return true;
  t->ok = true;
  return true;
}

static bool build_rows_analysis(Plan* p, RowsAnaTables* t, int W, int out_cols, const std::vector<float>& tab);
static bool build_rows_synthesis(Plan* p, RowsSynTables* t, int W, int in_cols, const std::vector<float>& tab);

bool fast_plan_init(Plan* p) {
  p->fast = nullptr;
  cudaDeviceProp prop{};
  if (!cuda_ok(cudaGetDeviceProperties(&prop, p->device), "cudaGetDeviceProperties")) return false;
  if (prop.major != 10) return true;   // tcgen05 path is sm_100-only
  FastTables* f = new FastTables();
  f->sm_count = prop.multiProcessorCount;
  {
    const DimTables& Ld = p->dim[p->d - 1];
    if (!build_rows_analysis(p, &f->rows_ana[0], Ld.N, 2 * Ld.k, p->h_TA) ||
        !build_rows_analysis(p, &f->rows_ana[1], Ld.M, 2 * Ld.k, p->h_TST) ||
        !build_rows_synthesis(p, &f->rows_syn[0], Ld.M, 2 * Ld.k, p->h_TS) ||
        !build_rows_synthesis(p, &f->rows_syn[1], Ld.N, 2 * Ld.k, p->h_TAT)) {
      delete f;
      return false;
    }
  }
  if (p->d < 2) { p->fast = f; return true; }   // only the tensor-core contraction applies to 1-D problems
  const DimTables& L = p->dim[p->d - 1];
  const DimTables& Y = p->dim[p->d - 2];
  bool good = build_fused_analysis(p, &f->ana[0], Y.N, L.N, Y.k, L.k, p->h_TA, Y.h_A) &&
              build_fused_analysis(p, &f->ana[1], Y.M, L.M, Y.k, L.k, p->h_TST, Y.h_SH) &&
              build_fused_synthesis(p, &f->syn[0], Y.M, L.M, Y.k, L.k, p->h_TS, Y.h_S) &&
              build_fused_synthesis(p, &f->syn[1], Y.N, L.N, Y.k, L.k, p->h_TAT, Y.h_AH);
  if (!good) { delete f; return false; }
  p->fast = f;
  return true;
}

void fast_plan_destroy(Plan* p) {
  delete p->fast;
  p->fast = nullptr;
}

// d == 2: the fused kernels are the whole transform.  d == 3: they handle the last two dims of every (image, z) slice and
// the generic complex table kernel handles dim 0 on the already-truncated data (sc_api.cu).
bool fast_can_analyze(const Plan* p, bool adjoint) {
  return p->fast != nullptr && (p->d == 2 || p->d == 3) && p->fast->ana[adjoint ? 1 : 0].ok;
}
bool fast_can_synthesize(const Plan* p, bool adjoint) {
  return p->fast != nullptr && (p->d == 2 || p->d == 3) && p->fast->syn[adjoint ? 1 : 0].ok;
}
int fast_tile_group(const Plan* p, bool synthesis, bool adjoint) {
  return synthesis ? p->fast->syn[adjoint ? 1 : 0].G : p->fast->ana[adjoint ? 1 : 0].G;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tensor_map_encoder() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}
// fp32 matrix [rows x W] (row-major), boxes of [32 rows x 32 floats], 128-byte swizzle
static bool make_row_tile_map(CUtensorMap* map, float* base, uint64_t rows, uint64_t W) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (enc == nullptr) { set_error("cuTensorMapEncodeTiled entry point not available"); return false; }
  const cuuint64_t dims[2] = {W, rows};
  const cuuint64_t strides[1] = {W * sizeof(float)};
  const cuuint32_t box[2] = {32, 32};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (row tiles) failed: CUresult " + std::to_string((int)r) + ", base " +
              std::to_string((unsigned long long)(uintptr_t)base) + ", rows " + std::to_string(rows) + ", W " + std::to_string(W));
    return false;
  }
  return true;
}

// fp32 matrix [rows x W] (row-major), boxes of [128 rows x 32 floats] in the 128-byte swizzle: a thread that owns a row reads
// its eight 16-byte chunks from eight different bank groups than its neighbours
static bool make_swizzled_box_map(CUtensorMap* map, const float* base, uint64_t rows, uint64_t W) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (enc == nullptr) { set_error("cuTensorMapEncodeTiled entry point not available"); return false; }
  const cuuint64_t dims[2] = {W, rows};
  const cuuint64_t strides[1] = {W * sizeof(float)};
  const cuuint32_t box[2] = {32, 128};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (swizzled x boxes) failed: CUresult " + std::to_string((int)r)); return false; }
  return true;
}

// fp32 matrix [rows x W] (row-major), boxes of [128 rows x 64 floats], no swizzle (the converters read 16-byte pieces)
static bool make_slab_load_map(CUtensorMap* map, const float* base, uint64_t rows, uint64_t W) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (enc == nullptr) { set_error("cuTensorMapEncodeTiled entry point not available"); return false; }
  const cuuint64_t dims[2] = {W, rows};
  const cuuint64_t strides[1] = {W * sizeof(float)};
  const cuuint32_t box[2] = {64, 128};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (x slabs) failed: CUresult " + std::to_string((int)r) + ", base " +
              std::to_string((unsigned long long)(uintptr_t)base) + ", rows " + std::to_string(rows) + ", W " + std::to_string(W));
    return false;
  }
  return true;
}

// 16-bit image matrix [rows x W] (row-major): kind 3 = x loads, boxes [128 rows x 64 elements] in the 128-byte swizzle
// (k_fused_analysis2); kind 4 = dx stores, boxes [32 rows x 32 elements] in the 64-byte swizzle (k_fused_synthesis)
static bool make_16bit_map(CUtensorMap* map, const void* base, uint64_t rows, uint64_t W, int storage, bool store) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (enc == nullptr) { set_error("cuTensorMapEncodeTiled entry point not available"); return false; }
  const cuuint64_t dims[2] = {W, rows};
  const cuuint64_t strides[1] = {W * 2};
  const cuuint32_t box[2] = {store ? 32u : 64u, store ? 32u : 128u};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(map, storage == SC_FLAG_GRID_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                         const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         store ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                         store ? CU_TENSOR_MAP_L2_PROMOTION_NONE : CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (16-bit images) failed: CUresult " + std::to_string((int)r)); return false; }
  return true;
}

// 3-D view {contiguous floats, second index, quads} of a quad-major tensor: one request per 1 KB row of the box
static bool cached_wide_map(const Plan* p, const float2* base, uint64_t inner_floats, uint64_t n_second, uint64_t nq, uint64_t stride_second_bytes,
                            uint64_t stride_quad_bytes, uint32_t box_inner, uint32_t box_second, CUtensorMap* out, uint32_t box_quads) {
  FastTables* f = p->fast;
  std::lock_guard<std::mutex> lock(f->map_mutex);
  // shares the gather cache: rows = inner_floats, k = n_second, sr = 0 marks the 3-D kind
  for (const GatherMapCacheEntry& e : f->gather_cache)
    if (e.base == base && e.nq == nq && e.rows == inner_floats && e.k == n_second && e.sq == stride_quad_bytes && e.sr == 0 &&
        e.sk == stride_second_bytes && e.box_rows == box_inner && e.box_k == box_second + (box_quads << 16)) { *out = e.map; return true; }
  if (!thread_has_context()) cudaFree(nullptr);   // (see cached_map)
  EncodeTiledFn enc = tensor_map_encoder();
  if (enc == nullptr) { set_error("cuTensorMapEncodeTiled entry point not available"); return false; }
  GatherMapCacheEntry e{base, nq, inner_floats, n_second, stride_quad_bytes, 0, stride_second_bytes, box_inner, box_second + (box_quads << 16), {}};
  const cuuint64_t dims[3] = {inner_floats, n_second, nq};
  const cuuint64_t strides[2] = {stride_second_bytes, stride_quad_bytes};
  const cuuint32_t box[3] = {box_inner, box_second, box_quads};
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUresult r = enc(&e.map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float2*>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (wide rows) failed: CUresult " + std::to_string((int)r)); return false; }
  if (f->gather_cache.size() >= 48) f->gather_cache.erase(f->gather_cache.begin());
  f->gather_cache.push_back(e);
  *out = e.map;
  return true;
}

// ---- probe: how fast does the TMA engine gather 32-byte sectors?  One CTA per quad of modes pulls its [Ci x Co x 32 B] block of a
// (Ci, Co, modes) complex64 tensor into shared memory with 4-D tensor loads (box {8 floats, 1 quad, 64 o, 8 i} = 16 KB), all eight
// boxes in flight at once; per-CTA cycles (start -> every box landed) go to `cycles_out`.
__global__ void __launch_bounds__(64) k_tma_gather_probe(const __grid_constant__ CUtensorMap w_map, long long* cycles_out, int n_boxes,
                                                         int k_per_box) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ uint64_t bar[16];
  if (threadIdx.x == 0) {
    for (int i = 0; i < n_boxes; ++i) mbar_init(&bar[i], 1);
    mbar_init_fence();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const long long t0 = clock64();
    for (int c = 0; c < n_boxes; ++c) {
      mbar_arrive_expect_tx(&bar[c], (uint32_t)(k_per_box * 64 * 32));
      tma_load_4d(smem + (size_t)c * k_per_box * 64 * 32, &w_map, &bar[c], 0, (int)blockIdx.x, 0, c * k_per_box);
    }
    const long long t1 = clock64();
    for (int c = 0; c < n_boxes; ++c) mbar_wait(&bar[c], 0);
    const long long t2 = clock64();
    cycles_out[2 * blockIdx.x] = t1 - t0;
    cycles_out[2 * blockIdx.x + 1] = t2 - t0;
  }
}

static bool make_sector_gather_map(CUtensorMap* map, const float2* base, uint64_t n_quads, uint64_t n_rows, uint64_t n_k,
                                   uint64_t stride_quad_bytes, uint64_t stride_row_bytes, uint64_t stride_k_bytes, uint32_t box_rows,
                                   uint32_t box_k);

bool tma_gather_probe(const float2* w, int Ci, int Co, int64_t Mt, long long* cycles_out, cudaStream_t st) {
  if (Mt % 4 != 0 || Ci % 8 != 0 || Ci > 128 || Co != 64) { set_error("tma probe: need Mt % 4 == 0, Co == 64, Ci % 8 == 0, Ci <= 128"); return false; }
  if (!thread_has_context()) cudaFree(nullptr);
  CUtensorMap map;
  if (!make_sector_gather_map(&map, w, (uint64_t)(Mt / 4), (uint64_t)Co, (uint64_t)Ci, 32, (uint64_t)Mt * 8, (uint64_t)Co * Mt * 8, 64, 8))
    return false;
  const int n_boxes = Ci / 8;
  const size_t smem = (size_t)n_boxes * 8 * 64 * 32 + 1024;
  if (!cuda_ok(cudaFuncSetAttribute(k_tma_gather_probe, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
               "cudaFuncSetAttribute(k_tma_gather_probe)"))
    return false;
  k_tma_gather_probe<<<(unsigned)(Mt / 4), 64, smem, st>>>(map, cycles_out, n_boxes, 8);
  count_launch();
  return cuda_ok(cudaGetLastError(), "k_tma_gather_probe launch");
}

// (quad, row, k) view of a complex64 tensor whose 4 consecutive modes are one 32-byte sector: dims {8 floats, quads, rows, k},
// box {8, 1, box_rows, box_k}: one tensor load gathers box_rows x box_k sectors into a dense [k][row][8 floats] block
static bool make_sector_gather_map(CUtensorMap* map, const float2* base, uint64_t n_quads, uint64_t n_rows, uint64_t n_k,
                                   uint64_t stride_quad_bytes, uint64_t stride_row_bytes, uint64_t stride_k_bytes, uint32_t box_rows,
                                   uint32_t box_k) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (enc == nullptr) { set_error("cuTensorMapEncodeTiled entry point not available"); return false; }
  const cuuint64_t dims[4] = {8, n_quads, n_rows, n_k};
  const cuuint64_t strides[3] = {stride_quad_bytes, stride_row_bytes, stride_k_bytes};
  const cuuint32_t box[4] = {8, 1, box_rows, box_k};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float2*>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (sector gather) failed: CUresult " + std::to_string((int)r));
    return false;
  }
  return true;
}

// launch with programmatic stream serialization: the kernel may begin (prologue only; see pdl_wait) before the previous
// kernel of the stream has drained
static cudaError_t launch_pdl(const void* func, dim3 grid, dim3 block, size_t smem, cudaStream_t st, void** args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelExC(&cfg, func, args);
}

// L2 evict-first policy on the image streams (x / gy loads, y / dx stores) so that the weights and mode tensors a step re-reads
// stay L2-resident.  Measured on B200 (round 2, cfg-2 graph step, two A/B pairs): 167.5k -> 169.4k samples/s.
// SC_L2_STREAM_HINT=0 switches it off at run time for A/B runs.
constexpr int SC_L2_STREAM_HINT_DEFAULT = 1;
static int l2_stream_hint_enabled() {
  static const int v = [] {
    const char* e = getenv("SC_L2_STREAM_HINT");
    return e != nullptr ? (atoi(e) != 0 ? 1 : 0) : SC_L2_STREAM_HINT_DEFAULT;
  }();
  return v;
}

// SC_TRACE_FILE=<path>: record the per-role timeline of CTA 0 of every fused transform launch (debug only; synchronises)
static long long* trace_begin() {
  if (getenv("SC_TRACE_FILE") == nullptr) return nullptr;
  long long* d = nullptr;
  if (cudaMalloc(&d, 8 * 16 * 4 * sizeof(long long)) != cudaSuccess) return nullptr;
  cudaMemset(d, 0, 8 * 16 * 4 * sizeof(long long));
  return d;
}
static void trace_end(long long* d, const char* what) {
  if (d == nullptr) return;
  std::vector<long long> h(8 * 16 * 4);
  cudaDeviceSynchronize();
  cudaMemcpy(h.data(), d, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
  cudaFree(d);
  FILE* f = fopen(getenv("SC_TRACE_FILE"), "a");
  if (f == nullptr) return;
  fprintf(f, "# %s\n", what);
  for (int r = 0; r < 8; ++r)
    for (int i = 0; i < 16; ++i)
      fprintf(f, "%d %d %lld %lld %lld\n", r, i, h[(r * 16 + i) * 4], h[(r * 16 + i) * 4 + 1], h[(r * 16 + i) * 4 + 2]);
  fclose(f);
}

static bool ana2_enabled() {
  static const bool on = [] { const char* e = getenv("SC_ANA2"); return e == nullptr || atoi(e) != 0; }();   // =0: first generation (A/B runs)
  return on;
}

bool fast_analysis_reads_16bit(const Plan* p) { return p->fast != nullptr && p->fast->ana[0].v2_ok && ana2_enabled(); }

bool fast_analyze(const Plan* p, const float* images, int64_t n_images, float2* modes_out, bool adjoint, cudaStream_t st,
                  bool quad_major, const L2Prefetch* pf, int storage) {
  const FusedAnalysisTables& t = p->fast->ana[adjoint ? 1 : 0];
  if (quad_major && ((t.KY * t.KX) % 4 != 0 || (reinterpret_cast<uintptr_t>(modes_out) & 31u) != 0)) {
    set_error("fast_analyze: the quad-major layout needs a mode count that is a multiple of 4 and a 32-byte aligned buffer");
    return false;
  }
  if (n_images % t.G != 0) { set_error("fast_analyze: image count not a multiple of the tile group"); return false; }
  AnaParams P{};
  P.x = images; P.out = modes_out; P.b1_img = t.d_b1; P.a2_img = t.d_a2;
  P.n_tiles = (int)(n_images / t.G); P.W = t.W; P.slabs = t.slabs; P.N1 = t.N1; P.KX = t.KX; P.QROWS = t.G * t.KY;
  P.n_stages = t.n_stages; P.tmem_cols = t.tmem_cols;
  P.l2_stream_hint = l2_stream_hint_enabled();
  P.quad_major = quad_major ? 1 : 0; P.G = t.G; P.Mt = t.KY * t.KX; P.n_images = n_images;
  if (pf != nullptr) {
    static const bool pf_on = [] { const char* e = getenv("SC_L2_PREFETCH"); return e == nullptr || atoi(e) != 0; }();   // =0: A/B runs
    for (int r = 0; r < 2 && pf_on; ++r) {
      if (pf->ptr[r] == nullptr || (reinterpret_cast<uintptr_t>(pf->ptr[r]) & 15u) != 0) continue;
      P.pf_ptr[r] = static_cast<const uint8_t*>(pf->ptr[r]);
      P.pf_bytes[r] = pf->bytes[r] & ~(unsigned long long)15;
    }
  }
  P.off_f32 = t.off_f32; P.off_ring = t.off_ring;
  P.off_b1 = t.off_b1; P.off_a2 = t.off_a2; P.off_b2 = t.off_b2; P.off_scratch = t.off_scratch; P.stage_off = t.stage_off;
  P.trace = trace_begin();
  const int grid = persistent_grid(p, P.n_tiles);
  CUtensorMap x_map;
  if (storage != 0 && (adjoint || !fast_analysis_reads_16bit(p))) { set_error("fast_analyze: 16-bit images need k_fused_analysis2"); return false; }
  if (t.v2_ok && ana2_enabled()) {
    P.n_stages = t.v2_stages; P.tmem_cols = 512;
    P.off_f32 = 0; P.off_ring = 0; P.off_b1 = t.v2_off_b1; P.off_a2 = t.v2_off_b2; P.off_b2 = t.v2_off_b2; P.off_scratch = t.v2_off_scratch;
    if (!cached_map(p, storage ? 3 : 2, images, (uint64_t)P.n_tiles * 128, (uint64_t)t.W, &x_map, storage)) return false;
    CUtensorMap qm_map = x_map;   // (placeholder when unused)
    static const bool qm_tma_on = [] { const char* e = getenv("SC_QM_TMA"); return e == nullptr || atoi(e) != 0; }();   // =0: store loop (A/B runs)
    if (quad_major && qm_tma_on && t.G == 1 && P.Mt / 4 <= 256 && ((P.off_scratch + P.stage_off) % 128u) == 0 && (P.Mt * 8) % 128 == 0) {
      // {8 floats, images, quads}: image stride 32 B, quad stride n_images * 32 B
      if (!cached_wide_map(p, modes_out, 8, (uint64_t)n_images, (uint64_t)(P.Mt / 4), 32, (uint64_t)n_images * 32, 8, 1, &qm_map, (uint32_t)(P.Mt / 4)))
        return false;
      P.qm_tma = 1;
    }
    switch (t.N1) {
#define SC_FA2_LAUNCH(N, S)                                                                                      \
  {                                                                                                              \
    static SmemOptIn opt_in;                                                                                     \
    if (!ensure_dynamic_smem((const void*)k_fused_analysis2<N, S>, opt_in, p->device, t.v2_smem_bytes,           \
                             "cudaFuncSetAttribute(k_fused_analysis2)")) return false;                          \
    void* args[] = {(void*)&P, (void*)&x_map, (void*)&qm_map};                                                 \
    if (!cuda_ok(launch_pdl((const void*)k_fused_analysis2<N, S>, dim3(grid), dim3(FA_THREADS), t.v2_smem_bytes, st, args), \
                 "k_fused_analysis2 launch")) return false;                                                     \
  }
#define SC_FA2_CASE(N)                                                                                           \
  case N:                                                                                                        \
    if (storage == SC_FLAG_GRID_F16) SC_FA2_LAUNCH(N, SC_FLAG_GRID_F16)                                          \
    else if (storage == SC_FLAG_GRID_BF16) SC_FA2_LAUNCH(N, SC_FLAG_GRID_BF16)                                   \
    else SC_FA2_LAUNCH(N, 0)                                                                                     \
    break;
      SC_FA2_CASE(16) SC_FA2_CASE(32) SC_FA2_CASE(48)
#undef SC_FA2_CASE
#undef SC_FA2_LAUNCH
      default: set_error("fast_analyze: unsupported N1"); return false;
    }
    count_launch();
    trace_end(P.trace, "analysis2");
    return cuda_ok(cudaGetLastError(), "k_fused_analysis2 launch");
  }
  if (!cached_map(p, 0, images, (uint64_t)P.n_tiles * 128, (uint64_t)t.W, &x_map)) return false;
  switch (t.N1) {
#define SC_FA_CASE(N)                                                                                            \
  case N: {                                                                                                      \
    static SmemOptIn opt_in;                                                                                     \
    if (!ensure_dynamic_smem((const void*)k_fused_analysis<N>, opt_in, p->device, t.smem_bytes,                  \
                             "cudaFuncSetAttribute(k_fused_analysis)")) return false;                           \
    { void* args[] = {(void*)&P, (void*)&x_map};                                                               \
      if (!cuda_ok(launch_pdl((const void*)k_fused_analysis<N>, dim3(grid), dim3(FA_THREADS), t.smem_bytes, st, args), \
                   "k_fused_analysis launch")) return false; }                                              \
  } break;
    SC_FA_CASE(16) SC_FA_CASE(32) SC_FA_CASE(48) SC_FA_CASE(64)
#undef SC_FA_CASE
    default: set_error("fast_analyze: unsupported N1"); return false;
  }
  count_launch();
  trace_end(P.trace, "analysis");
  return cuda_ok(cudaGetLastError(), "k_fused_analysis launch");
}

bool fast_synthesize(const Plan* p, const float2* modes_in, int64_t n_images, int n_channels, const float* bias,
                     float* images_out, bool adjoint, int slices_per_image, cudaStream_t st, bool quad_major, int storage) {
  const FusedSynthesisTables& t = p->fast->syn[adjoint ? 1 : 0];
  if (storage != 0 && (!adjoint || bias != nullptr)) { set_error("fast_synthesize: 16-bit output is the adjoint synthesis (dx) only"); return false; }
  if (quad_major && (t.KY * t.KX) % 4 != 0) { set_error("fast_synthesize: the quad-major layout needs a mode count that is a multiple of 4"); return false; }
  if (n_images % t.G != 0) { set_error("fast_synthesize: image count not a multiple of the tile group"); return false; }
  SynParams P{};
  P.modes = modes_in; P.out = images_out; P.bias = bias; P.aa_img = t.d_aa; P.bb_img = t.d_bb;
  P.n_tiles = (int)(n_images / t.G); P.W = t.W; P.KX = t.KX; P.QROWS = t.G * t.KY; P.H = t.H;
  P.n_channels = n_channels > 0 ? n_channels : 1; P.tmem_cols = t.tmem_cols;
  P.slices_per_image = slices_per_image > 0 ? slices_per_image : 1;
  P.quad_major = quad_major ? 1 : 0; P.KY = t.KY; P.n_images = n_images;
  static const int syn_hint = [] { const char* e = getenv("SC_SYN_STORE_HINT"); return e == nullptr ? -1 : atoi(e); }();   // A/B runs
  P.l2_stream_hint = syn_hint >= 0 ? syn_hint : l2_stream_hint_enabled();
  P.off_aa = t.off_aa; P.off_ba = t.off_ba; P.off_u = t.off_u; P.off_bb = t.off_bb; P.off_stage = t.off_stage;
  P.trace = trace_begin();
  const int grid = persistent_grid(p, P.n_tiles);
  CUtensorMap out_map;
  if (!cached_map(p, storage ? 4 : 1, images_out, (uint64_t)P.n_tiles * 128, (uint64_t)t.W, &out_map, storage)) return false;
  switch (t.N1) {
#define SC_FS_LAUNCH(N, S)                                                                                       \
  {                                                                                                              \
    static SmemOptIn opt_in;                                                                                     \
    if (!ensure_dynamic_smem((const void*)k_fused_synthesis<N, S>, opt_in, p->device, t.smem_bytes,              \
                             "cudaFuncSetAttribute(k_fused_synthesis)")) return false;                          \
    void* args[] = {(void*)&P, (void*)&out_map};                                                               \
    if (!cuda_ok(launch_pdl((const void*)k_fused_synthesis<N, S>, dim3(grid), dim3(FS_THREADS), t.smem_bytes, st, args), \
                 "k_fused_synthesis launch")) return false;                                                     \
  }
#define SC_FS_CASE(N)                                                                                            \
  case N:                                                                                                        \
    if (storage == SC_FLAG_GRID_F16) SC_FS_LAUNCH(N, SC_FLAG_GRID_F16)                                           \
    else if (storage == SC_FLAG_GRID_BF16) SC_FS_LAUNCH(N, SC_FLAG_GRID_BF16)                                    \
    else SC_FS_LAUNCH(N, 0)                                                                                      \
    break;
    SC_FS_CASE(16) SC_FS_CASE(32) SC_FS_CASE(48) SC_FS_CASE(64)
#undef SC_FS_CASE
#undef SC_FS_LAUNCH
    default: set_error("fast_synthesize: unsupported N1"); return false;
  }
  count_launch();
  trace_end(P.trace, "synthesis");
  return cuda_ok(cudaGetLastError(), "k_fused_synthesis launch");
}

// =====================================================================================================
// "rows" kernels: the last-dim transform alone on tensor cores, for ANY number of rows
//
//   Validated on B200 in round 2 (tests/test_gpu_rows.py); SC_ROWS=0 switches them off at run time for A/B runs.
//
//   The fused 2-D kernels above need a whole image inside one 128-row tile (H <= 128, W <= 128/256).  Larger grids (cfg-5:
//   256^2 .. 1024^2), 1-D problems and 3-D problems with big planes run the generic chain: a real table GEMM over the last dim,
//   which touches > 90 % of the bytes, then complex table products on the already-truncated leading dims.  These two kernels
//   replace only that last-dim step; rows are whatever the leading dims multiply out to (a multiple of 128).
//
//   rows-analysis   C[r, 0:2k] = sum_w X[r, w] * T[w, 0:2k]           M = 128 rows, N = 2*N1 (T1 | T2), K = W in 64-column slabs
//     warp 13     TMA producer: x slab [128 x 64] fp32 -> staging ring; table slab [2*N1 x 64] bf16 image (pre-swizzled, L2
//                 resident, <= 32 KB) -> the operand ring slot, by a 1-D bulk copy
//     warps 5-12  converters: staging -> bf16 hi/lo -> swizzled operand slab           (same code as the fused kernel)
//     warp 4      MMA issuer (+ TMEM allocation): D[buf] += x_hi*[T1;T2] + x_lo*T1
//     warps 0-3   epilogue: D -> (hi + lo sums) -> the row's 2k floats in global memory
//   rows-synthesis  Y[r, w] = sum_j U[r, j] * T[j, w] (+ bias)          M = 128 rows, N = 64-column chunks, K = N1 <= 128
//     warp 9      producer: the tile's contiguous [128 x 2k] fp32 block -> staging (one bulk copy); table chunk images
//                 [T1 | T2] x [64 columns x K] -> two-deep ring
//     warps 5-8   prep: staging row -> bf16 hi/lo A operand (single buffer)
//     warp 4      MMA issuer: D[buf] = U_hi*T1 + U_lo*T1 + U_hi*T2 per chunk
//     warps 0-3   epilogue: D -> + bias -> swizzled [32 x 32] boxes -> TMA tensor stores      (same code as the fused kernel)
// =====================================================================================================
constexpr int RA_CONV_WARPS = 8;
constexpr int RA_CONV_WARP0 = 5;
constexpr int RA_TMA_WARP = RA_CONV_WARP0 + RA_CONV_WARPS;   // 13
constexpr int RA_THREADS = (RA_TMA_WARP + 1) * 32;           // 448
constexpr int RA_CONV_ITERS = 128 / (RA_CONV_WARPS * 2);
constexpr int RA_MAX_F32 = 3, RA_MAX_RING = 4;

struct RowsAnaParams {
  float* out;               // [rows x out_cols] fp32
  const uint8_t* tab_img;   // per 64-column slab of the input: [2*N1 rows x 64] bf16 SW128 image (T1 rows, then T2 rows)
  int n_tiles, slabs, out_cols, f32_stages, ring_stages, tmem_cols;
  uint32_t off_f32, off_ring, slot_bytes, tab_bytes;
};

template <int N1>
__global__ void __launch_bounds__(RA_THREADS, 1) k_rows_analysis(const RowsAnaParams P, const __grid_constant__ CUtensorMap x_map) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ uint64_t bar_f32_full[RA_MAX_F32], bar_f32_empty[RA_MAX_F32], bar_full[RA_MAX_RING], bar_tab_full[RA_MAX_RING],
      bar_empty[RA_MAX_RING], bar_d_full[2], bar_d_empty[2];
  __shared__ uint32_t tmem_base_slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int NS = P.ring_stages, FS = P.f32_stages;
  if (tid == 0) {
    for (int i = 0; i < FS; ++i) { mbar_init(&bar_f32_full[i], 1); mbar_init(&bar_f32_empty[i], RA_CONV_WARPS); }
    for (int i = 0; i < NS; ++i) { mbar_init(&bar_full[i], RA_CONV_WARPS); mbar_init(&bar_tab_full[i], 1); mbar_init(&bar_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_d_full[i], 1); mbar_init(&bar_d_empty[i], 128); }
    mbar_init_fence();
  }
  if (warp == 4) tmem_alloc(&tmem_base_slot, (uint32_t)P.tmem_cols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = tmem_base_slot;
  const uint32_t tm_d[2] = {tmem, tmem + (uint32_t)(2 * N1)};
  const int n_local = (P.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int total = n_local * P.slabs;

  if (warp == RA_TMA_WARP) {
    // ------------------------------------------------------------------ producer
    uint8_t* f32_stage = smem + P.off_f32;
    pdl_wait();                                  // x is produced by the previous kernel of the stream
    pdl_launch_dependents();                     // (after the wait: see k_fused_analysis)
    for (int idx = 0; idx < total; ++idx) {
      const int sb = idx % FS;
      const int tile = (int)blockIdx.x + (idx / P.slabs) * (int)gridDim.x, slab = idx % P.slabs;
      mbar_wait(&bar_f32_empty[sb], (uint32_t)(((idx / FS) & 1) ^ 1));
      if (elect_one()) {
        mbar_arrive_expect_tx(&bar_f32_full[sb], 32768u);
        tma_load_2d(f32_stage + sb * 32768, &x_map, &bar_f32_full[sb], slab * 64, tile * 128);
      }
      __syncwarp();
      const int slot = idx % NS;
      mbar_wait(&bar_empty[slot], (uint32_t)(((idx / NS) & 1) ^ 1));   // the MMAs that read this slot two rounds ago are done
      if (elect_one()) {
        mbar_arrive_expect_tx(&bar_tab_full[slot], P.tab_bytes);
        bulk_load_1d(smem + P.off_ring + (size_t)slot * P.slot_bytes + 32768u, P.tab_img + (size_t)slab * P.tab_bytes, P.tab_bytes,
                     &bar_tab_full[slot]);
      }
      __syncwarp();
    }
  } else if (warp >= RA_CONV_WARP0) {
    // ------------------------------------------------------------------ converters (fp32 staging -> bf16 hi/lo operand slabs)
    const int lt = tid - RA_CONV_WARP0 * 32;
    constexpr int RP = RA_CONV_WARPS * 2;        // rows covered per pass
    const int rbase = lt >> 4, c4 = lt & 15;     // 16 float4 per 64-float row segment
    uint8_t* f32_stage = smem + P.off_f32;
    const uint32_t my_f32 = (uint32_t)(rbase * 256 + c4 * 16);
    for (int idx = 0; idx < total; ++idx) {
      const int slot = idx % NS;
      const uint32_t ph = (uint32_t)((idx / NS) & 1);
      const int sb = idx % FS;
      mbar_wait(&bar_f32_full[sb], (uint32_t)((idx / FS) & 1));
      uint2 hi[RA_CONV_ITERS], lo[RA_CONV_ITERS];
      const uint8_t* fsrc = f32_stage + sb * 32768 + my_f32;
#pragma unroll
      for (int it = 0; it < RA_CONV_ITERS; ++it) {
        const float4 v = *reinterpret_cast<const float4*>(fsrc + it * RP * 256);
        split2_bf16(v.x, v.y, hi[it].x, lo[it].x);
        split2_bf16(v.z, v.w, hi[it].y, lo[it].y);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_f32_empty[sb]);
      mbar_wait(&bar_empty[slot], ph ^ 1u);
      uint8_t* shi = smem + P.off_ring + (size_t)slot * P.slot_bytes;
      uint8_t* slo = shi + FA_SLAB_BYTES;
#pragma unroll
      for (int it = 0; it < RA_CONV_ITERS; ++it) {
        const uint32_t off = sw128_offset(rbase + it * RP, c4 * 4, 128);
        *reinterpret_cast<uint2*>(shi + off) = hi[it];
        *reinterpret_cast<uint2*>(slo + off) = lo[it];
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_full[slot]);
    }
  } else if (warp == 4) {
    // ------------------------------------------------------------------ MMA issuer
    const uint32_t idesc_p1 = idesc_bf16(128, 2 * N1), idesc_p2 = idesc_bf16(128, N1);
    const uint32_t ring_lo = desc_lo(smem_u32(smem + P.off_ring));
    int g = 0;
    for (int i = 0; i < n_local; ++i) {
      const int buf = i & 1;
      mbar_wait(&bar_d_empty[buf], (uint32_t)(((i >> 1) & 1) ^ 1));
      tc_fence_after_sync();
      for (int s = 0; s < P.slabs; ++s, ++g) {
        const int slot = g % NS;
        const uint32_t ph = (uint32_t)((g / NS) & 1);
        mbar_wait(&bar_full[slot], ph);
        mbar_wait(&bar_tab_full[slot], ph);
        tc_fence_after_sync();
        const uint32_t d_hi = ring_lo + (uint32_t)slot * (P.slot_bytes >> 4), d_lo = d_hi + (FA_SLAB_BYTES >> 4);
        const uint32_t d_b = d_hi + (32768u >> 4);
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            mma_bf16_ss(tm_d[buf], desc_from_lo(d_hi + 2 * kk), desc_from_lo(d_b + 2 * kk), idesc_p1, (s | kk) != 0);
            mma_bf16_ss(tm_d[buf], desc_from_lo(d_lo + 2 * kk), desc_from_lo(d_b + 2 * kk), idesc_p2, true);
          }
          mma_commit(&bar_empty[slot]);
        }
        __syncwarp();
      }
      if (elect_one()) mma_commit(&bar_d_full[buf]);
      __syncwarp();
    }
  } else {
    // ------------------------------------------------------------------ epilogue: D -> the row's out_cols floats
    const int row = warp * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(warp * 32) << 16;
    const int oc = P.out_cols;
    pdl_wait();                                  // the output buffer may still be read by the previous kernel
    for (int i = 0; i < n_local; ++i) {
      const int buf = i & 1;
      const int tile = (int)blockIdx.x + i * (int)gridDim.x;
      float* dst = P.out + ((size_t)tile * 128 + row) * oc;
      mbar_wait(&bar_d_full[buf], (uint32_t)((i >> 1) & 1));
      tc_fence_after_sync();
#pragma unroll
      for (int c = 0; c < N1; c += 16) {
        float t1[16], t2[16];
        tmem_ld16(tm_d[buf] + lane_sel + c, t1);        // x_hi*T1 + x_lo*T1
        tmem_ld16(tm_d[buf] + lane_sel + N1 + c, t2);   // x_hi*T2
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 16; e += 2)
          if (c + e < oc) *reinterpret_cast<float2*>(dst + c + e) = make_float2(t1[e] + t2[e], t1[e + 1] + t2[e + 1]);
      }
      tc_fence_before_sync();
      mbar_arrive(&bar_d_empty[buf]);
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem, (uint32_t)P.tmem_cols);
}

constexpr int RS_PREP_WARP0 = 5, RS_PREP_WARPS = 4, RS_TMA_WARP = RS_PREP_WARP0 + RS_PREP_WARPS;   // 9
constexpr int RS_THREADS = (RS_TMA_WARP + 1) * 32;                                                  // 320

struct RowsSynParams {
  const float* u;           // [rows x in_cols] fp32 (re, im interleaved)
  const float* bias;        // may be null
  const uint8_t* tab_img;   // per 64-column chunk of the output: T1 image then T2 image, each [64 rows x KS*64] bf16 SW128
  int n_tiles, in_cols, n_chunks, n_channels, tmem_cols;
  long long rows_per_image;
  uint32_t off_a, off_ustage, off_tab, off_stage, u_bytes, chunk_bytes;
};

template <int N1>
__global__ void __launch_bounds__(RS_THREADS, 1) k_rows_synthesis(const RowsSynParams P, const __grid_constant__ CUtensorMap out_map) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ uint64_t bar_u_full, bar_u_empty, bar_a_full, bar_a_empty, bar_tab_full[2], bar_tab_empty[2], bar_d_full[2], bar_d_empty[2];
  __shared__ uint32_t tmem_base_slot;
  constexpr int KS = (N1 + 63) / 64;                    // K slabs of the A operand / of a table image
  constexpr uint32_t A_HALF = (uint32_t)KS * FA_SLAB_BYTES;   // hi slabs, then lo slabs
  constexpr uint32_t T_IMG = (uint32_t)KS * 8192u;      // one [64 x KS*64] table image
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    mbar_init(&bar_u_full, 1);  mbar_init(&bar_u_empty, RS_PREP_WARPS);
    mbar_init(&bar_a_full, RS_PREP_WARPS);  mbar_init(&bar_a_empty, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bar_tab_full[i], 1); mbar_init(&bar_tab_empty[i], 1);
      mbar_init(&bar_d_full[i], 1);   mbar_init(&bar_d_empty[i], 128);
    }
    mbar_init_fence();
  }
  if (warp == 4) tmem_alloc(&tmem_base_slot, (uint32_t)P.tmem_cols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = tmem_base_slot;
  const uint32_t tm_d[2] = {tmem, tmem + 64u};
  const int n_local = (P.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int NCH = P.n_chunks;

  if (warp == RS_TMA_WARP) {
    // ------------------------------------------------------------------ producer
    pdl_wait();                                  // U is produced by the previous kernel of the stream
    pdl_launch_dependents();                     // (after the wait: see k_fused_analysis)
    int gc = 0;
    for (int i = 0; i < n_local; ++i) {
      const int tile = (int)blockIdx.x + i * (int)gridDim.x;
      mbar_wait(&bar_u_empty, (uint32_t)((i & 1) ^ 1));
      if (elect_one()) {
        mbar_arrive_expect_tx(&bar_u_full, P.u_bytes);
        bulk_load_1d(smem + P.off_ustage, P.u + (size_t)tile * 128 * P.in_cols, P.u_bytes, &bar_u_full);
      }
      __syncwarp();
      for (int c = 0; c < NCH; ++c, ++gc) {
        const int slot = gc & 1;
        mbar_wait(&bar_tab_empty[slot], (uint32_t)(((gc >> 1) & 1) ^ 1));
        if (elect_one()) {
          mbar_arrive_expect_tx(&bar_tab_full[slot], P.chunk_bytes);
          bulk_load_1d(smem + P.off_tab + (size_t)slot * P.chunk_bytes, P.tab_img + (size_t)c * P.chunk_bytes, P.chunk_bytes,
                       &bar_tab_full[slot]);
        }
        __syncwarp();
      }
    }
  } else if (warp >= RS_PREP_WARP0) {
    // ------------------------------------------------------------------ prep: staging row -> bf16 hi/lo A operand
    const int r = tid - RS_PREP_WARP0 * 32;      // tile row
    const float* urow = reinterpret_cast<const float*>(smem + P.off_ustage) + (size_t)r * P.in_cols;
    uint8_t* arow = smem + P.off_a + r * 128;
    const int ic = P.in_cols;
    for (int i = 0; i < n_local; ++i) {
      mbar_wait(&bar_u_full, (uint32_t)(i & 1));
      mbar_wait(&bar_a_empty, (uint32_t)((i & 1) ^ 1));   // the MMAs of the previous tile have read the operand
#pragma unroll
      for (int c0 = 0; c0 < N1 / 8; ++c0) {
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; e += 2) {
          const int j = 8 * c0 + e;                        // in_cols is even: a pair is inside or outside together
          const float2 pr = j < ic ? *reinterpret_cast<const float2*>(urow + j) : make_float2(0.f, 0.f);
          v[e] = pr.x; v[e + 1] = pr.y;
        }
        uint32_t hw[4], lw[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) split2_bf16(v[2 * e], v[2 * e + 1], hw[e], lw[e]);
        uint8_t* dst = arow + (c0 >> 3) * FA_SLAB_BYTES + ((((c0 & 7) ^ r) & 7) << 4);
        *reinterpret_cast<uint4*>(dst) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
        *reinterpret_cast<uint4*>(dst + A_HALF) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) { mbar_arrive(&bar_a_full); mbar_arrive(&bar_u_empty); }
    }
  } else if (warp == 4) {
    // ------------------------------------------------------------------ MMA issuer
    const uint32_t idesc = idesc_bf16(128, 64);
    const uint32_t a_lo0 = desc_lo(smem_u32(smem + P.off_a)), tab_lo0 = desc_lo(smem_u32(smem + P.off_tab));
    int gc = 0;
    for (int i = 0; i < n_local; ++i) {
      mbar_wait(&bar_a_full, (uint32_t)(i & 1));
      tc_fence_after_sync();
      for (int c = 0; c < NCH; ++c, ++gc) {
        const int slot = gc & 1;
        const uint32_t ph = (uint32_t)((gc >> 1) & 1);
        mbar_wait(&bar_tab_full[slot], ph);
        mbar_wait(&bar_d_empty[slot], ph ^ 1u);
        tc_fence_after_sync();
        const uint32_t t1 = tab_lo0 + (uint32_t)slot * (P.chunk_bytes >> 4), t2 = t1 + (T_IMG >> 4);
        if (elect_one()) {
#pragma unroll
          for (int ks = 0; ks < N1 / 16; ++ks) {
            const uint32_t a_hi = a_lo0 + (uint32_t)(ks >> 2) * (FA_SLAB_BYTES >> 4) + 2 * (ks & 3), a_lo = a_hi + (A_HALF >> 4);
            const uint32_t b_off = (uint32_t)(ks >> 2) * (8192u >> 4) + 2 * (ks & 3);
            mma_bf16_ss(tm_d[slot], desc_from_lo(a_hi), desc_from_lo(t1 + b_off), idesc, ks > 0);
            mma_bf16_ss(tm_d[slot], desc_from_lo(a_lo), desc_from_lo(t1 + b_off), idesc, true);
            mma_bf16_ss(tm_d[slot], desc_from_lo(a_hi), desc_from_lo(t2 + b_off), idesc, true);
          }
          mma_commit(&bar_tab_empty[slot]);
          mma_commit(&bar_d_full[slot]);
          if (c == NCH - 1) mma_commit(&bar_a_empty);
        }
        __syncwarp();
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue: D -> + bias -> TMA tensor stores
    const int row = warp * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(warp * 32) << 16;
    uint8_t* my_stage = smem + P.off_stage + warp * 8192;   // two [32 x 128 B] boxes per warp
    uint32_t box_ctr = 0;
    int gc = 0;
    pdl_wait();                                             // the output image may still be read by the previous kernel
    for (int i = 0; i < n_local; ++i) {
      const int tile = (int)blockIdx.x + i * (int)gridDim.x;
      float b = 0.f;
      if (P.bias != nullptr) b = __ldg(P.bias + (int)((((long long)tile * 128 + row) / P.rows_per_image) % P.n_channels));
      for (int c = 0; c < NCH; ++c, ++gc) {
        const int buf = gc & 1;
        mbar_wait(&bar_d_full[buf], (uint32_t)((gc >> 1) & 1));
        tc_fence_after_sync();
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          float t[2][16];
          tmem_ld16(tm_d[buf] + lane_sel + 32 * hf, t[0]);
          tmem_ld16(tm_d[buf] + lane_sel + 32 * hf + 16, t[1]);
          uint8_t* box = my_stage + (box_ctr & 1) * 4096;
          if (lane == 0) bulk_wait_read_1();        // the store issued two boxes ago has finished reading this buffer
          __syncwarp();
          tmem_ld_wait();
#pragma unroll
          for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int e = 0; e < 16; e += 4) {
              const int ch = (16 * u + e) >> 2;      // 16-byte chunk index within the 128-byte row
              *reinterpret_cast<float4*>(box + lane * 128 + (((ch ^ lane) & 7) << 4)) =
                  make_float4(t[u][e] + b, t[u][e + 1] + b, t[u][e + 2] + b, t[u][e + 3] + b);
            }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&out_map, box, c * 64 + 32 * hf, tile * 128 + warp * 32);
            bulk_commit();
          }
          ++box_ctr;
        }
        tc_fence_before_sync();
        mbar_arrive(&bar_d_empty[buf]);
      }
    }
    if (lane == 0) bulk_wait_all();
    __syncwarp();
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem, (uint32_t)P.tmem_cols);
}

// ---- host side --------------------------------------------------------------------------------------
static bool rows_kernels_enabled() {
  static const bool on = [] { const char* e = getenv("SC_ROWS"); return e == nullptr || atoi(e) != 0; }();
  return on;
}

// `tab` is [W x out_cols] row-major (p->h_TA / p->h_TST)
static bool build_rows_analysis(Plan* p, RowsAnaTables* t, int W, int out_cols, const std::vector<float>& tab) {
  t->ok = false;
  if (W % 64 != 0 || out_cols < 2 || out_cols > 128) return true;
  const int N1 = ((out_cols + 15) / 16) * 16;
  t->W = W; t->N1 = N1; t->out_cols = out_cols; t->slabs = W / 64;
  t->tab_bytes = (uint32_t)(2 * N1 * 128);
  t->slot_bytes = 32768u + t->tab_bytes;
  t->tmem_cols = 4 * N1 <= 64 ? 64 : 4 * N1 <= 128 ? 128 : 4 * N1 <= 256 ? 256 : 512;
  const uint32_t budget = 227u * 1024u - 4096u;
  t->ring_stages = 2;
  t->f32_stages = 3;
  if ((uint32_t)t->f32_stages * 32768u + 2u * t->slot_bytes + 1024u > budget) t->f32_stages = 2;
  if ((uint32_t)t->f32_stages * 32768u + 2u * t->slot_bytes + 1024u > budget) return true;
  t->off_f32 = 0;
  t->off_ring = (uint32_t)t->f32_stages * 32768u;
  t->smem_bytes = t->off_ring + 2u * t->slot_bytes + 1024u;
  // every slab is its own [2*N1 x 64] image: host_sw128_offset puts slab s at s * rows * 128 bytes
  std::vector<uint8_t> img((size_t)t->slabs * t->tab_bytes, 0);
  for (int j = 0; j < out_cols; ++j)
    for (int w = 0; w < W; ++w) put_split(img, 2 * N1, j, N1 + j, w, tab[(size_t)w * out_cols + j]);
  if (!upload_bytes(p, img, &t->d_tab)) return false;
  t->ok = true;
  return true;
}

// `tab` is [in_cols x W] row-major (p->h_TS / p->h_TAT)
static bool build_rows_synthesis(Plan* p, RowsSynTables* t, int W, int in_cols, const std::vector<float>& tab) {
  t->ok = false;
  if (W % 64 != 0 || in_cols < 2 || in_cols > 128) return true;
  const int N1 = ((in_cols + 15) / 16) * 16;
  const int KS = (N1 + 63) / 64;
  t->W = W; t->N1 = N1; t->in_cols = in_cols; t->n_chunks = W / 64;
  t->tmem_cols = 128;
  t->u_bytes = (uint32_t)(128 * in_cols * 4);
  t->chunk_bytes = (uint32_t)(2 * KS * 8192);
  t->off_a = 0;
  t->off_ustage = (uint32_t)(2 * KS) * (uint32_t)FA_SLAB_BYTES;
  t->off_tab = t->off_ustage + ((t->u_bytes + 1023u) & ~1023u);
  t->off_stage = t->off_tab + 2u * t->chunk_bytes;
  t->smem_bytes = t->off_stage + 4u * 8192u + 1024u;
  if (t->smem_bytes > 227u * 1024u - 4096u) return true;
  std::vector<uint8_t> img((size_t)t->n_chunks * t->chunk_bytes, 0);
  for (int c = 0; c < t->n_chunks; ++c)
    for (int n = 0; n < 64; ++n)
      for (int j = 0; j < in_cols; ++j) {
        const float v = tab[(size_t)j * W + c * 64 + n];
        const uint16_t t1 = bf16_bits(v);
        const uint16_t t2 = bf16_bits(v - bf16_to_float(t1));
        const size_t base = (size_t)c * t->chunk_bytes + host_sw128_offset(n, j, 64);
        memcpy(&img[base], &t1, 2);
        memcpy(&img[base + (size_t)KS * 8192], &t2, 2);
      }
  if (!upload_bytes(p, img, &t->d_tab)) return false;
  t->ok = true;
  return true;
}

bool rows_can_analyze(const Plan* p, bool adjoint, int64_t rows) {
  return rows_kernels_enabled() && p->fast != nullptr && p->fast->rows_ana[adjoint ? 1 : 0].ok && rows > 0 && rows % 128 == 0;
}
bool rows_can_synthesize(const Plan* p, bool adjoint, int64_t rows) {
  return rows_kernels_enabled() && p->fast != nullptr && p->fast->rows_syn[adjoint ? 1 : 0].ok && rows > 0 && rows % 128 == 0;
}

bool rows_analyze(const Plan* p, const float* x, int64_t rows, float* out, bool adjoint, cudaStream_t st) {
  const RowsAnaTables& t = p->fast->rows_ana[adjoint ? 1 : 0];
  RowsAnaParams P{};
  P.out = out; P.tab_img = t.d_tab;
  P.n_tiles = (int)(rows / 128); P.slabs = t.slabs; P.out_cols = t.out_cols;
  P.f32_stages = t.f32_stages; P.ring_stages = t.ring_stages; P.tmem_cols = t.tmem_cols;
  P.off_f32 = t.off_f32; P.off_ring = t.off_ring; P.slot_bytes = t.slot_bytes; P.tab_bytes = t.tab_bytes;
  const int grid = persistent_grid(p, P.n_tiles);
  CUtensorMap x_map;
  if (!cached_map(p, 0, x, (uint64_t)rows, (uint64_t)t.W, &x_map)) return false;
  switch (t.N1) {
#define SC_RA_CASE(N)                                                                                            \
  case N: {                                                                                                      \
    static SmemOptIn opt_in;                                                                                     \
    if (!ensure_dynamic_smem((const void*)k_rows_analysis<N>, opt_in, p->device, t.smem_bytes,                   \
                             "cudaFuncSetAttribute(k_rows_analysis)")) return false;                            \
    { void* args[] = {(void*)&P, (void*)&x_map};                                                               \
      if (!cuda_ok(launch_pdl((const void*)k_rows_analysis<N>, dim3(grid), dim3(RA_THREADS), t.smem_bytes, st, args), \
                   "k_rows_analysis launch")) return false; }                                               \
  } break;
    SC_RA_CASE(16) SC_RA_CASE(32) SC_RA_CASE(48) SC_RA_CASE(64) SC_RA_CASE(80) SC_RA_CASE(96) SC_RA_CASE(112) SC_RA_CASE(128)
#undef SC_RA_CASE
    default: set_error("rows_analyze: unsupported N1"); return false;
  }
  count_launch();
  return cuda_ok(cudaGetLastError(), "k_rows_analysis launch");
}

bool rows_synthesize(const Plan* p, const float* u, int64_t rows, float* out, const float* bias, int64_t rows_per_image,
                     int n_channels, bool adjoint, cudaStream_t st) {
  const RowsSynTables& t = p->fast->rows_syn[adjoint ? 1 : 0];
  RowsSynParams P{};
  P.u = u; P.bias = bias; P.tab_img = t.d_tab;
  P.n_tiles = (int)(rows / 128); P.in_cols = t.in_cols; P.n_chunks = t.n_chunks;
  P.n_channels = n_channels > 0 ? n_channels : 1; P.tmem_cols = t.tmem_cols;
  P.rows_per_image = rows_per_image > 0 ? rows_per_image : 1;
  P.off_a = t.off_a; P.off_ustage = t.off_ustage; P.off_tab = t.off_tab; P.off_stage = t.off_stage;
  P.u_bytes = t.u_bytes; P.chunk_bytes = t.chunk_bytes;
  const int grid = persistent_grid(p, P.n_tiles);
  CUtensorMap out_map;
  if (!cached_map(p, 1, out, (uint64_t)rows, (uint64_t)t.W, &out_map)) return false;
  switch (t.N1) {
#define SC_RS_CASE(N)                                                                                            \
  case N: {                                                                                                      \
    static SmemOptIn opt_in;                                                                                     \
    if (!ensure_dynamic_smem((const void*)k_rows_synthesis<N>, opt_in, p->device, t.smem_bytes,                  \
                             "cudaFuncSetAttribute(k_rows_synthesis)")) return false;                           \
    { void* args[] = {(void*)&P, (void*)&out_map};                                                             \
      if (!cuda_ok(launch_pdl((const void*)k_rows_synthesis<N>, dim3(grid), dim3(RS_THREADS), t.smem_bytes, st, args), \
                   "k_rows_synthesis launch")) return false; }                                              \
  } break;
    SC_RS_CASE(16) SC_RS_CASE(32) SC_RS_CASE(48) SC_RS_CASE(64) SC_RS_CASE(80) SC_RS_CASE(96) SC_RS_CASE(112) SC_RS_CASE(128)
#undef SC_RS_CASE
    default: set_error("rows_synthesize: unsupported N1"); return false;
  }
  count_launch();
  return cuda_ok(cudaGetLastError(), "k_rows_synthesis launch");
}

}  // namespace sc
