// Internal plan object shared by the translation units of libspectral_conv_b200.so.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "spectral_conv_b200.h"

namespace sc {

// One spatial dimension of the problem.  Host vectors mirror the device tables.
struct DimTables {
  int N = 0;       // input grid
  int M = 0;       // output grid
  int F = 0;       // spectrum length on the input grid
  int k = 0;       // kept modes
  int w0 = 0;      // first weight row used
  std::vector<int> in_bins;  // unshifted bin per kept slot
  std::vector<int> out_bins; // bin of the OUTPUT grid the slot is synthesised at (-1: dropped); == in_bins unless SC_FLAG_RESAMPLE
  // leading dims only: complex tables, row-major, interleaved (re,im)
  float2* d_A = nullptr;    // analysis          [k x N]   exp(-2 pi i b n / N)
  float2* d_AH = nullptr;   // its adjoint       [N x k]
  float2* d_S = nullptr;    // synthesis         [M x k]   exp(+2 pi i b n / M) * [b < M]
  float2* d_SH = nullptr;   // its adjoint       [k x M]
  std::vector<float2> h_A, h_AH, h_S, h_SH;   // host copies (the fast path derives its bf16 operand images from them)
};

struct FastTables;   // sc_fast.cu

struct Plan {
  sc_problem prob{};
  int device = 0;
  int d = 0;
  DimTables dim[SC_MAX_DIMS];
  int64_t n_modes_total = 1;   // prod k_j
  int64_t grid_points = 1;     // prod N_j
  int64_t out_points = 1;      // prod M_j
  double s_fwd = 1.0, s_inv = 1.0;
  int dc_slot = 0;             // flat index of the all-zero-frequency slot inside the kept block
  // last dim: real tables, row-major, row length padded to `ld` floats
  float* d_TA = nullptr;  int ldTA = 0;    // analysis            [N_d x 2k]  (cos, -sin) * s_fwd
  float* d_TAT = nullptr; int ldTAT = 0;   // adjoint of analysis [2k x N_d]
  float* d_TS = nullptr;  int ldTS = 0;    // synthesis           [2k x M_d]  Hermitian rules, * s_inv
  float* d_TST = nullptr; int ldTST = 0;   // adjoint of synthesis[M_d x 2k]
  int32_t* d_woff = nullptr;               // weight element offset of kept mode m (complex elements)
  int64_t weight_elems_per_io = 1;         // prod max_n_modes
  bool weight_block_is_whole = true;       // kept block == whole weight tensor
  bool fast_enabled = true;
  int reserved_sms = 0;                    // SMs the persistent transform kernels leave free (for a concurrent collective)
  bool host_only = false;                  // tables computed on the host only, nothing uploaded (sc_problem_table)
  int grid16 = 0;                          // SC_FLAG_GRID_F16 / SC_FLAG_GRID_BF16: storage of x / dx, 0 = float
  std::vector<float> h_TA, h_TAT, h_TS, h_TST;   // host copies of the last-dim tables
  FastTables* fast = nullptr;              // tcgen05 path state (nullptr when the shape does not qualify)
  std::vector<void*> owned;                // every cudaMalloc made for this plan
};

void set_error(const std::string& msg);
bool cuda_ok(cudaError_t e, const char* what);
extern std::atomic<uint64_t> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

// ---- generic SIMT kernels (sc_generic.cu) -----------------------------------------------------------
// C[R x Nc] = A[R x Kc] * T[Kc x ldt] (+ bias[(r / rows_per_image) % n_channels])
bool launch_real_table_gemm(const float* A, const float* T, int ldt, float* C, const float* bias,
                            int64_t R, int Kc, int Nc, int64_t rows_per_image, int n_channels, cudaStream_t st);
// out[o, p, i] = sum_q T[p, q] * in[o, q, i]   (complex; T is [P x Q] row-major)
bool launch_complex_table_gemm(const float2* T, const float2* in, float2* out, int64_t O, int P, int Q, int I,
                               cudaStream_t st);
bool launch_complex_table_gemm_strided(const float2* T, int64_t sTp, int64_t sTq, bool conjT, const float2* in, float2* out,
                                       int64_t O, int P, int Q, int I, cudaStream_t st);
// out[p, q] (strided) = sum_{o,i} conj(A[o,p,i]) * B[o,q,i]
bool launch_pair_reduce(const float2* A, const float2* B, float2* out, int64_t sOp, int64_t sOq, int64_t O, int P, int Q, int I,
                        cudaStream_t st);
// CP pieces (sc_generic.cu, section 2c)
bool launch_cp_scale(const float2* const* u, const int* k, int d, const float2* lambda, float2* scale, int R, int64_t M, cudaStream_t st);
bool launch_cp_apply(const float2* in, const float2* scale, float2* out, bool conj_scale, int batch, int64_t per_batch, cudaStream_t st);
bool launch_cp_dscale(const float2* t, const float2* g, float2* dscale, int batch, int64_t per_batch, cudaStream_t st);
bool launch_cp_factor_grad(const float2* const* u, const int* k, int d, const float2* lambda, const float2* dscale, float2* out,
                           int which, int R, int64_t M, cudaStream_t st);
// out[r, c, m] = sum_k opA(A[r,k,m]) * opB(B[k,c,m]); per-operand element strides, optional mode-offset tables
struct ModeGemmOperand {
  const void* ptr; int64_t s_outer; int64_t s_inner; const int32_t* mode_off;  // mode_off == nullptr -> m itself
};
bool launch_mode_gemm(ModeGemmOperand A, bool conjA, ModeGemmOperand B, bool conjB, ModeGemmOperand Out,
                      int nR, int nC, int nK, int64_t nModes, cudaStream_t st);
bool launch_bias_grad(const float2* gm, float* dbias, int batch, int out_channels, int64_t n_modes, int dc_slot,
                      float inv_scale, cudaStream_t st);
// 16-bit image storage (grid16 = SC_FLAG_GRID_F16 / SC_FLAG_GRID_BF16): n elements 16-bit -> float (to_16 false) or float -> 16-bit
// rounded to nearest even (to_16 true)
bool launch_grid_convert(int grid16, const void* in, void* out, int64_t n, bool to_16, cudaStream_t st);

// two-shot all-reduce (average) over NVLink peer memory, sc_collective.cu
bool launch_allreduce_p2p(float* const* bufs, uint32_t* const* signals, int rank, int world, int64_t n_floats, float scale, int n_ctas,
                          cudaStream_t st);

}  // namespace sc
