// tcgen05 / TMA fused transform path (sc_fast.cu): interface seen by the orchestration in sc_api.cu.
#pragma once
#include "sc_plan.h"

#define SC_STR_(x) #x
#define SC_STR(x) SC_STR_(x)

namespace sc {

bool fast_plan_init(Plan* p);       // builds the fast-path tables when the shape qualifies; false only on CUDA errors
void fast_plan_destroy(Plan* p);
bool fast_can_analyze(const Plan* p, bool adjoint);
bool fast_can_synthesize(const Plan* p, bool adjoint);
// quad_major: the mode tensor is laid out [quad of 4 modes][image][4] instead of [image][modes] -- an internal layout of the dense
// forward / backward chains: every operand access of the tensor-core contraction becomes contiguous along the image index
// up to two contiguous global ranges the analysis launch pulls into L2 for the kernels that follow it (see AnaParams)
struct L2Prefetch { const void* ptr[2] = {nullptr, nullptr}; unsigned long long bytes[2] = {0, 0}; };
// storage: 0 = float images, SC_FLAG_GRID_F16 / SC_FLAG_GRID_BF16 = 16-bit images (the `float*` then addresses 16-bit data):
// the forward analysis reads x that way when fast_analysis_reads_16bit(p), the adjoint synthesis writes dx that way
bool fast_analyze(const Plan* p, const float* images, int64_t n_images, float2* modes_out, bool adjoint,
                  cudaStream_t st, bool quad_major = false, const L2Prefetch* prefetch = nullptr, int storage = 0);
bool fast_analysis_reads_16bit(const Plan* p);
// n_images counts the 2-D slices the fused kernel sees (images x dim-0 extent for 3-D problems)
bool fast_synthesize(const Plan* p, const float2* modes_in, int64_t n_images, int n_channels, const float* bias,
                     float* images_out, bool adjoint, int slices_per_image, cudaStream_t st, bool quad_major = false,
                     int storage = 0);
int fast_tile_group(const Plan* p, bool synthesis, bool adjoint);   // slices per 128-row tile

void fast_set_reserve(bool on);   // the next persistent transform launches of this thread leave plan->reserved_sms SMs free
bool quad2_enabled();   // second-generation quad contraction kernel selected (default; SC_QUAD=1 selects the first)
bool mode_gemm_quad_eligible(const Plan* p, int64_t n_modes, const void* a, const void* b, const void* out);
bool fast_can_contract(const Plan* p, int B, int Ci, int Co, bool quad_ok);
// optional extras of a tensor-core contraction launch
struct ModeGemmExtras {
  bool a_early = false, b_early = false;   // the operand is NOT written by the kernel launched just before on the stream:
                                           // its loads may start ahead of the grid-dependency wait
  bool l2_resident = false;                // both operands are expected in L2 already: no prefetch instructions
  long long sAQ = 0, sBQ = 0, sOQ = 0;     // quad strides of a / b / out when they are in the quad-major layout (0: standard layout)
  float* dbias = nullptr; float bias_scale = 1.f;   // dweight launch only (b = gm): also dbias[o] = scale * sum_b Re gm[b, o, DC]
  bool bias_done = false;                  // out: the launch computed dbias
};
// out[R, n] (+ per-mode offset) = sum_k a(R, k) * b(n, k), complex, one product per kept mode, on tcgen05 (bf16x3)
bool launch_mode_gemm_tc(const Plan* p, const float2* a, long long sAR, long long sAK, const int* offA, bool conjA,
                         const float2* b, long long sBN, long long sBK, const int* offB, float2* out, long long sOR,
                         long long sON, const int* offO, int MR, int NB, int KC, int64_t n_modes, cudaStream_t st,
                         ModeGemmExtras* extras = nullptr);
// last-dim transform alone on tensor cores for any number of rows (multiple of 128); see the end of sc_fast.cu
bool rows_can_analyze(const Plan* p, bool adjoint, int64_t rows);
bool rows_can_synthesize(const Plan* p, bool adjoint, int64_t rows);
bool rows_analyze(const Plan* p, const float* x, int64_t rows, float* out, bool adjoint, cudaStream_t st);
bool rows_synthesize(const Plan* p, const float* u, int64_t rows, float* out, const float* bias, int64_t rows_per_image,
                     int n_channels, bool adjoint, cudaStream_t st);
bool tma_gather_probe(const float2* w, int Ci, int Co, int64_t Mt, long long* cycles_out, cudaStream_t st);
bool umma_selftest_ts(const float* A, const float* B, float* D, int N, int K, cudaStream_t st);
bool umma_selftest(const float* A, const float* B, float* D, int N, int K, cudaStream_t st);

}  // namespace sc
