// Generic (any grid size, any mode count, 1..4-D) SIMT fp32 kernels of the SpectralConv path.
//
// The truncated transforms are expressed as products with small precomputed twiddle tables, so odd grids,
// odd mode counts, resampled outputs and the Hermitian rules of the reference's C2R step
// (spectral_convolution.py:552-559) are all properties of the table, not of the kernel.  The tcgen05/TMA
// path (sc_fast_*.cu) covers the large power-of-two shapes; this file is the path every other shape takes
// and the cross-check for the fast one.  Compiled for sm_100a only.
#include <algorithm>

#include "sc_half.cuh"
#include "sc_plan.h"

namespace sc {

// =====================================================================================================
// 1. real table GEMM:   C[R x Nc] = A[R x Kc] * T[Kc x ldt]   (+ per-channel bias)
//    analysis of the last dim  (Kc = N_d,  Nc = 2 k_d)   and   synthesis of the last dim (Kc = 2 k_d, Nc = M_d)
// =====================================================================================================
constexpr int RG_BM = 128;      // rows per CTA
constexpr int RG_BK = 32;       // k-chunk
constexpr int RG_THREADS = 256; // 8 column-groups x 32 row-groups, 4 rows x TN cols per thread

template <int TN>
__device__ __forceinline__ void rg_step(float (&acc)[4][TN], const float (&As)[RG_BM][RG_BK + 1],
                                        const float (&Ts)[RG_BK][8 * TN], int ty, int tx, int k) {
  float a[4], t[TN];
#pragma unroll
  for (int m = 0; m < 4; ++m) a[m] = As[ty * 4 + m][k];
#pragma unroll
  for (int n = 0; n < TN; ++n) t[n] = Ts[k][tx * TN + n];
#pragma unroll
  for (int m = 0; m < 4; ++m)
#pragma unroll
    for (int n = 0; n < TN; ++n) acc[m][n] = fmaf(a[m], t[n], acc[m][n]);
}

template <int TN>
__global__ void __launch_bounds__(RG_THREADS)
k_real_table_gemm(const float* __restrict__ A, const float* __restrict__ T, int ldt, float* __restrict__ C,
                  const float* __restrict__ bias, long long R, int Kc, int Nc, long long rows_per_image,
                  int n_channels) {
  constexpr int BN = 8 * TN;
  __shared__ float As[RG_BM][RG_BK + 1];
  __shared__ float Ts[RG_BK][BN];
  const int tx = threadIdx.x & 7;
  const int ty = threadIdx.x >> 3;
  const long long row0 = (long long)blockIdx.x * RG_BM;
  const int col0 = blockIdx.y * BN;

  float acc[4][TN];
#pragma unroll
  for (int m = 0; m < 4; ++m)
#pragma unroll
    for (int n = 0; n < TN; ++n) acc[m][n] = 0.f;

  for (int k0 = 0; k0 < Kc; k0 += RG_BK) {
    // A tile: a warp reads 32 consecutive floats of one row (128 B, coalesced)
#pragma unroll 4
    for (int idx = threadIdx.x; idx < RG_BM * RG_BK; idx += RG_THREADS) {
      const int r = idx / RG_BK, k = idx % RG_BK;
      const long long gr = row0 + r;
      float v = 0.f;
      if (gr < R && k0 + k < Kc) v = __ldg(A + gr * (long long)Kc + k0 + k);
      As[r][k] = v;
    }
    for (int idx = threadIdx.x; idx < RG_BK * BN; idx += RG_THREADS) {
      const int k = idx / BN, c = idx % BN;
      float v = 0.f;
      if (k0 + k < Kc && col0 + c < ldt) v = __ldg(T + (long long)(k0 + k) * ldt + col0 + c);
      Ts[k][c] = v;
    }
    __syncthreads();
    if (k0 + RG_BK <= Kc) {
#pragma unroll
      for (int k = 0; k < RG_BK; ++k) rg_step<TN>(acc, As, Ts, ty, tx, k);
    } else {   // ragged tail of the contraction (e.g. Kc = 2 k_d = 34): do not multiply the zero padding
      const int kmax = Kc - k0;
#pragma unroll 2
      for (int k = 0; k < kmax; ++k) rg_step<TN>(acc, As, Ts, ty, tx, k);
    }
    __syncthreads();
  }

#pragma unroll
  for (int m = 0; m < 4; ++m) {
    const long long gr = row0 + ty * 4 + m;
    if (gr >= R) continue;
    float b = 0.f;
    if (bias != nullptr) b = __ldg(bias + (gr / rows_per_image) % n_channels);
#pragma unroll
    for (int n = 0; n < TN; ++n) {
      const int gc = col0 + tx * TN + n;
      if (gc < Nc) C[gr * (long long)Nc + gc] = acc[m][n] + b;
    }
  }
}

template <int TN>
static void launch_rg(const float* A, const float* T, int ldt, float* C, const float* bias, int64_t R, int Kc,
                      int Nc, int64_t rows_per_image, int n_channels, int n_tiles, cudaStream_t st) {
  dim3 grid((unsigned)((R + RG_BM - 1) / RG_BM), (unsigned)n_tiles);
  k_real_table_gemm<TN><<<grid, RG_THREADS, 0, st>>>(A, T, ldt, C, bias, (long long)R, Kc, Nc,
                                                      (long long)rows_per_image, n_channels);
}

bool launch_real_table_gemm(const float* A, const float* T, int ldt, float* C, const float* bias, int64_t R,
                            int Kc, int Nc, int64_t rows_per_image, int n_channels, cudaStream_t st) {
  if (R <= 0 || Nc <= 0) return true;
  // split Nc into equal column tiles of at most 96 columns, 8 column-groups of TN each
  const int n_tiles = (Nc + 95) / 96;
  const int per_tile = (Nc + n_tiles - 1) / n_tiles;
  const int tn = (per_tile + 7) / 8;
#define SC_RG_CASE(N) \
  case N: launch_rg<N>(A, T, ldt, C, bias, R, Kc, Nc, rows_per_image, n_channels, (Nc + 8 * N - 1) / (8 * N), st); break;
  switch (tn) {
    SC_RG_CASE(1) SC_RG_CASE(2) SC_RG_CASE(3) SC_RG_CASE(4) SC_RG_CASE(5) SC_RG_CASE(6)
    SC_RG_CASE(7) SC_RG_CASE(8) SC_RG_CASE(9) SC_RG_CASE(10) SC_RG_CASE(11) SC_RG_CASE(12)
    default: set_error("real_table_gemm: internal tile selection failed"); return false;
  }
#undef SC_RG_CASE
  count_launch();
  return cuda_ok(cudaGetLastError(), "k_real_table_gemm launch");
}

// =====================================================================================================
// 2. complex table GEMM over a middle axis:   out[o, p, i] = sum_q T[p, q] * in[o, q, i]
//    (leading-dim analysis: Q = N_j, P = k_j;   leading-dim synthesis: Q = k_j, P = M_j)
//    lanes run over the flattened (o, i) columns, each thread owns CT_TP output rows of one column.
// =====================================================================================================
constexpr int CT_COLS = 128;   // columns per CTA (threadIdx.x)
constexpr int CT_TP = 16;      // output rows per thread
constexpr int CT_PG = 2;       // row groups per CTA (threadIdx.y)
constexpr int CT_QC = 32;      // q-chunk held in shared memory

template <bool CONJ_T>
__global__ void __launch_bounds__(CT_COLS* CT_PG)
k_complex_table_gemm(const float2* __restrict__ T, long long sTp, long long sTq, const float2* __restrict__ in,
                     float2* __restrict__ out, long long O, int P, int Q, int I) {
  __shared__ float2 s_in[CT_QC][CT_COLS];
  __shared__ __align__(16) float2 s_T[CT_QC][CT_PG * CT_TP + 2];   // +2: keeps rows 16-B aligned, spreads banks
  const long long ncols = O * (long long)I;
  const long long col = (long long)blockIdx.x * CT_COLS + threadIdx.x;
  const bool col_ok = col < ncols;
  const long long o = col_ok ? col / I : 0;
  const int i = col_ok ? (int)(col - o * I) : 0;
  const int p_base = blockIdx.y * (CT_PG * CT_TP);
  const int tid = threadIdx.y * CT_COLS + threadIdx.x;

  float2 acc[CT_TP];
#pragma unroll
  for (int t = 0; t < CT_TP; ++t) acc[t] = make_float2(0.f, 0.f);

  const float2* in_col = in + (o * Q) * (long long)I + i;
  for (int q0 = 0; q0 < Q; q0 += CT_QC) {
    for (int qq = threadIdx.y; qq < CT_QC; qq += CT_PG) {
      float2 v = make_float2(0.f, 0.f);
      if (col_ok && q0 + qq < Q) v = __ldg(in_col + (long long)(q0 + qq) * I);
      s_in[qq][threadIdx.x] = v;
    }
    for (int idx = tid; idx < CT_QC * CT_PG * CT_TP; idx += CT_COLS * CT_PG) {
      const int pp = idx / CT_QC, qq = idx % CT_QC;   // consecutive threads walk q: contiguous in T
      float2 v = make_float2(0.f, 0.f);
      if (p_base + pp < P && q0 + qq < Q) v = __ldg(T + (long long)(p_base + pp) * sTp + (long long)(q0 + qq) * sTq);
      if (CONJ_T) v.y = -v.y;
      s_T[qq][pp] = v;
    }
    __syncthreads();
#pragma unroll 4
    for (int qq = 0; qq < CT_QC; ++qq) {
      const float2 v = s_in[qq][threadIdx.x];
      const float4* trow = reinterpret_cast<const float4*>(&s_T[qq][threadIdx.y * CT_TP]);
#pragma unroll
      for (int t = 0; t < CT_TP / 2; ++t) {
        const float4 w = trow[t];   // two twiddles, warp-uniform address -> broadcast
        acc[2 * t].x = fmaf(w.x, v.x, acc[2 * t].x);
        acc[2 * t].x = fmaf(-w.y, v.y, acc[2 * t].x);
        acc[2 * t].y = fmaf(w.x, v.y, acc[2 * t].y);
        acc[2 * t].y = fmaf(w.y, v.x, acc[2 * t].y);
        acc[2 * t + 1].x = fmaf(w.z, v.x, acc[2 * t + 1].x);
        acc[2 * t + 1].x = fmaf(-w.w, v.y, acc[2 * t + 1].x);
        acc[2 * t + 1].y = fmaf(w.z, v.y, acc[2 * t + 1].y);
        acc[2 * t + 1].y = fmaf(w.w, v.x, acc[2 * t + 1].y);
      }
    }
    __syncthreads();
  }
  if (!col_ok) return;
  float2* out_col = out + (o * P) * (long long)I + i;
#pragma unroll
  for (int t = 0; t < CT_TP; ++t) {
    const int p = p_base + threadIdx.y * CT_TP + t;
    if (p < P) out_col[(long long)p * I] = acc[t];
  }
}

bool launch_complex_table_gemm_strided(const float2* T, int64_t sTp, int64_t sTq, bool conjT, const float2* in, float2* out,
                                       int64_t O, int P, int Q, int I, cudaStream_t st) {
  const int64_t ncols = O * (int64_t)I;
  if (ncols <= 0 || P <= 0) return true;
  dim3 grid((unsigned)((ncols + CT_COLS - 1) / CT_COLS), (unsigned)((P + CT_PG * CT_TP - 1) / (CT_PG * CT_TP)));
  dim3 block(CT_COLS, CT_PG);
  if (conjT)
    k_complex_table_gemm<true><<<grid, block, 0, st>>>(T, (long long)sTp, (long long)sTq, in, out, (long long)O, P, Q, I);
  else
    k_complex_table_gemm<false><<<grid, block, 0, st>>>(T, (long long)sTp, (long long)sTq, in, out, (long long)O, P, Q, I);
  count_launch();
  return cuda_ok(cudaGetLastError(), "k_complex_table_gemm launch");
}

bool launch_complex_table_gemm(const float2* T, const float2* in, float2* out, int64_t O, int P, int Q, int I,
                               cudaStream_t st) {
  return launch_complex_table_gemm_strided(T, Q, 1, false, in, out, O, P, Q, I, st);
}

// =====================================================================================================
// 2b. pair reduction (factor gradients of the factorized contractions):
//     out[p, q] = sum_{o, i} conj(A[o, p, i]) * B[o, q, i]        A: [O x P x I], B: [O x Q x I], out: P x Q (strided)
//     One CTA owns a 4 x 4 tile of `out`; its 256 threads stride over the flattened (o, i) reduction axis (consecutive
//     threads -> consecutive i: coalesced), then a warp-shuffle tree and a cross-warp pass in shared memory finish the sum.
// =====================================================================================================
constexpr int PR_T = 4;
constexpr int PR_THREADS = 512;
constexpr int PR_UNROLL = 2;    // reduction elements per thread and trip: 2 x 8 independent 64-bit loads in flight

__global__ void __launch_bounds__(PR_THREADS)
k_pair_reduce(const float2* __restrict__ A, const float2* __restrict__ B, float2* __restrict__ out, long long sOp,
              long long sOq, long long O, int P, int Q, int I) {
  __shared__ float2 s_part[PR_THREADS / 32][PR_T * PR_T];
  const int p0 = blockIdx.x * PR_T, q0 = blockIdx.y * PR_T;
  const long long R = O * (long long)I;
  float2 acc[PR_T][PR_T];
#pragma unroll
  for (int a = 0; a < PR_T; ++a)
#pragma unroll
    for (int b = 0; b < PR_T; ++b) acc[a][b] = make_float2(0.f, 0.f);
  // rows of the tile that exist (clamped rows re-read a valid row and are dropped at the store)
  int pa[PR_T], qb[PR_T];
#pragma unroll
  for (int a = 0; a < PR_T; ++a) { pa[a] = min(p0 + a, P - 1); qb[a] = min(q0 + a, Q - 1); }
  // (o, i) of this thread's element, advanced incrementally (no 64-bit division in the loop)
  long long o = threadIdx.x / I;
  int i = threadIdx.x - (int)o * I;
  const int step_o = PR_THREADS / I, step_i = PR_THREADS - step_o * I;
  for (long long r = threadIdx.x; r < R; r += (long long)PR_THREADS * PR_UNROLL) {
    float2 av[PR_UNROLL][PR_T], bv[PR_UNROLL][PR_T];
    bool ok[PR_UNROLL];
#pragma unroll
    for (int u = 0; u < PR_UNROLL; ++u) {
      ok[u] = r + (long long)u * PR_THREADS < R;
      const long long oo = ok[u] ? o : 0;
      const int ii = ok[u] ? i : 0;
#pragma unroll
      for (int a = 0; a < PR_T; ++a) {
        av[u][a] = __ldg(A + (oo * P + pa[a]) * (long long)I + ii);
        bv[u][a] = __ldg(B + (oo * Q + qb[a]) * (long long)I + ii);
      }
      o += step_o; i += step_i;
      if (i >= I) { i -= I; ++o; }
    }
#pragma unroll
    for (int u = 0; u < PR_UNROLL; ++u) {
      if (!ok[u]) continue;
#pragma unroll
      for (int a = 0; a < PR_T; ++a)
#pragma unroll
        for (int b = 0; b < PR_T; ++b) {   // conj(a) * b
          acc[a][b].x = fmaf(av[u][a].x, bv[u][b].x, acc[a][b].x);
          acc[a][b].x = fmaf(av[u][a].y, bv[u][b].y, acc[a][b].x);
          acc[a][b].y = fmaf(av[u][a].x, bv[u][b].y, acc[a][b].y);
          acc[a][b].y = fmaf(-av[u][a].y, bv[u][b].x, acc[a][b].y);
        }
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int a = 0; a < PR_T; ++a)
#pragma unroll
    for (int b = 0; b < PR_T; ++b) {
      float2 v = acc[a][b];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        v.x += __shfl_xor_sync(0xffffffffu, v.x, off);
        v.y += __shfl_xor_sync(0xffffffffu, v.y, off);
      }
      if (lane == 0) s_part[warp][a * PR_T + b] = v;
    }
  __syncthreads();
  if (threadIdx.x < PR_T * PR_T) {
    float2 v = make_float2(0.f, 0.f);
#pragma unroll
    for (int w = 0; w < PR_THREADS / 32; ++w) { v.x += s_part[w][threadIdx.x].x; v.y += s_part[w][threadIdx.x].y; }
    const int a = threadIdx.x / PR_T, b = threadIdx.x % PR_T;
    if (p0 + a < P && q0 + b < Q) out[(long long)(p0 + a) * sOp + (long long)(q0 + b) * sOq] = v;
  }
}

bool launch_pair_reduce(const float2* A, const float2* B, float2* out, int64_t sOp, int64_t sOq, int64_t O, int P, int Q,
                        int I, cudaStream_t st) {
  if (P <= 0 || Q <= 0) return true;
  dim3 grid((unsigned)((P + PR_T - 1) / PR_T), (unsigned)((Q + PR_T - 1) / PR_T));
  k_pair_reduce<<<grid, PR_THREADS, 0, st>>>(A, B, out, (long long)sOp, (long long)sOq, (long long)O, P, Q, I);
  count_launch();
  return cuda_ok(cudaGetLastError(), "k_pair_reduce launch");
}

// =====================================================================================================
// 2c. CP (canonical polyadic) pieces, reference `_contract_cp` :55-73.
//     scale[e, m] = lambda_e * prod_j U_j[m_j, e]   (Khatri-Rao rows of the kept mode-factor rows)
//     apply:  out[a, e, m] = in[a, e, m] * op(scale[e, m])
//     dscale[e, m] = sum_a conj(t[a, e, m]) * g[a, e, m]
//     factor gradients from dscale (warp per output element, shuffle reduction over the other mode indices)
// =====================================================================================================
struct CpFactors {
  const float2* u[SC_MAX_DIMS];   // [k_j x R] row-major, kept rows only
  int k[SC_MAX_DIMS];
  int d;
};

__device__ __forceinline__ float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__device__ __forceinline__ float2 cmul_conj_a(float2 a, float2 b) { return make_float2(a.x * b.x + a.y * b.y, a.x * b.y - a.y * b.x); }

// product over the mode factors except `skip` (skip = -1: all) for rank e and flat mode index m
__device__ __forceinline__ float2 cp_mode_product(const CpFactors& F, int R, int e, long long m, int skip) {
  float2 p = make_float2(1.f, 0.f);
  for (int j = F.d - 1; j >= 0; --j) {
    const int mj = (int)(m % F.k[j]);
    m /= F.k[j];
    if (j != skip) p = cmul(p, __ldg(F.u[j] + (long long)mj * R + e));
  }
  return p;
}

__global__ void k_cp_scale(CpFactors F, const float2* __restrict__ lambda, float2* __restrict__ scale, int R, long long M) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)R * M) return;
  const int e = (int)(idx / M);
  const long long m = idx - (long long)e * M;
  scale[idx] = cmul(__ldg(lambda + e), cp_mode_product(F, R, e, m, -1));
}

template <bool CONJ>
__global__ void k_cp_apply(const float2* __restrict__ in, const float2* __restrict__ scale, float2* __restrict__ out,
                           long long per_batch, long long total) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  float2 s = __ldg(scale + idx % per_batch);
  if (CONJ) s.y = -s.y;
  out[idx] = cmul(__ldg(in + idx), s);
}

__global__ void k_cp_dscale(const float2* __restrict__ t, const float2* __restrict__ g, float2* __restrict__ dscale,
                            int batch, long long per_batch) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= per_batch) return;
  float2 acc = make_float2(0.f, 0.f);
  for (int a = 0; a < batch; ++a) {
    const float2 v = cmul_conj_a(__ldg(t + a * per_batch + idx), __ldg(g + a * per_batch + idx));
    acc.x += v.x; acc.y += v.y;
  }
  dscale[idx] = acc;
}

// which == -1: dlambda[e] = sum_m conj(prod_j U_j) dscale[e,m]
// which == j : dU_j[r, e] = sum_{m : m_j == r} conj(lambda_e prod_{l != j} U_l) dscale[e,m]
// one warp per output element
__global__ void k_cp_factor_grad(CpFactors F, const float2* __restrict__ lambda, const float2* __restrict__ dscale,
                                 float2* __restrict__ out, int which, int R, long long M) {
  const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const long long n_out = which < 0 ? R : (long long)F.k[which] * R;
  if (w >= n_out) return;
  const int e = (int)(w % R);
  const int r = (int)(w / R);
  float2 acc = make_float2(0.f, 0.f);
  if (which < 0) {
    for (long long m = lane; m < M; m += 32) {
      const float2 v = cmul_conj_a(cp_mode_product(F, R, e, m, -1), __ldg(dscale + (long long)e * M + m));
      acc.x += v.x; acc.y += v.y;
    }
  } else {
    // enumerate the modes whose index along `which` equals r: m = (outer * k_which + r) * inner + i
    long long inner = 1, outer = 1;
    for (int j = which + 1; j < F.d; ++j) inner *= F.k[j];
    for (int j = 0; j < which; ++j) outer *= F.k[j];
    const float2 lam = __ldg(lambda + e);
    for (long long t = lane; t < outer * inner; t += 32) {
      const long long o = t / inner, i = t - o * inner;
      const long long m = (o * F.k[which] + r) * inner + i;
      const float2 coef = cmul(lam, cp_mode_product(F, R, e, m, which));
      const float2 v = cmul_conj_a(coef, __ldg(dscale + (long long)e * M + m));
      acc.x += v.x; acc.y += v.y;
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    acc.x += __shfl_xor_sync(0xffffffffu, acc.x, off);
    acc.y += __shfl_xor_sync(0xffffffffu, acc.y, off);
  }
  if (lane == 0) out[w] = acc;
}

static CpFactors make_cp_factors(const float2* const* u, const int* k, int d) {
  CpFactors F{};
  F.d = d;
  for (int j = 0; j < d; ++j) { F.u[j] = u[j]; F.k[j] = k[j]; }
  return F;
}

bool launch_cp_scale(const float2* const* u, const int* k, int d, const float2* lambda, float2* scale, int R, int64_t M,
                     cudaStream_t st) {
  const long long total = (long long)R * M;
  if (total <= 0) return true;
  k_cp_scale<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(make_cp_factors(u, k, d), lambda, scale, R, (long long)M);
  count_launch();
  return cuda_ok(cudaGetLastError(), "k_cp_scale launch");
}

bool launch_cp_apply(const float2* in, const float2* scale, float2* out, bool conj_scale, int batch, int64_t per_batch,
                     cudaStream_t st) {
  const long long total = (long long)batch * per_batch;
  if (total <= 0) return true;
  const unsigned grid = (unsigned)((total + 255) / 256);
  if (conj_scale) k_cp_apply<true><<<grid, 256, 0, st>>>(in, scale, out, (long long)per_batch, total);
  else k_cp_apply<false><<<grid, 256, 0, st>>>(in, scale, out, (long long)per_batch, total);
  count_launch();
  return cuda_ok(cudaGetLastError(), "k_cp_apply launch");
}

bool launch_cp_dscale(const float2* t, const float2* g, float2* dscale, int batch, int64_t per_batch, cudaStream_t st) {
  if (per_batch <= 0) return true;
  k_cp_dscale<<<(unsigned)((per_batch + 255) / 256), 256, 0, st>>>(t, g, dscale, batch, (long long)per_batch);
  count_launch();
  return cuda_ok(cudaGetLastError(), "k_cp_dscale launch");
}

bool launch_cp_factor_grad(const float2* const* u, const int* k, int d, const float2* lambda, const float2* dscale,
                           float2* out, int which, int R, int64_t M, cudaStream_t st) {
  const long long n_out = which < 0 ? R : (long long)k[which] * R;
  if (n_out <= 0) return true;
  const long long threads = n_out * 32;
  k_cp_factor_grad<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(make_cp_factors(u, k, d), lambda, dscale, out, which, R,
                                                                      (long long)M);
  count_launch();
  return cuda_ok(cudaGetLastError(), "k_cp_factor_grad launch");
}

// =====================================================================================================
// 3. mode-wise complex GEMM:  out[r, c, m] = sum_k opA(A[r, k, m]) * opB(B[k, c, m])
//    forward  : r=b c=o k=i   A = xm            B = weight
//    dxm      : r=b c=i k=o   A = gm            B = conj(weight) (strides swapped)
//    dweight  : r=i c=o k=b   A = conj(xm)      B = gm
//    lanes run over modes (the contiguous axis of every operand); a warp owns a TR x TC tile.
// =====================================================================================================
constexpr int MG_TR = 4;
constexpr int MG_TC = 8;
constexpr int MG_WARPS = 8;

struct MgOp {
  const float2* ptr;
  long long s_outer, s_inner;
  const int* off;
};

template <bool CONJ_A, bool CONJ_B>
__global__ void __launch_bounds__(32 * MG_WARPS, 2)
k_mode_gemm(MgOp A, MgOp B, float2* __restrict__ outp, long long so_r, long long so_c, const int* __restrict__ out_off,
            int nR, int nC, int nK, long long nModes) {
  const long long m = (long long)blockIdx.x * 32 + threadIdx.x;
  const int tiles_r = (nR + MG_TR - 1) / MG_TR;
  const int tiles_c = (nC + MG_TC - 1) / MG_TC;
  const int tile = blockIdx.y * MG_WARPS + threadIdx.y;   // r-tiles fastest: warps of a CTA share the B tile
  if (tile >= tiles_r * tiles_c || m >= nModes) return;
  const int r0 = (tile % tiles_r) * MG_TR;
  const int c0 = (tile / tiles_r) * MG_TC;
  const long long ma = A.off ? (long long)__ldg(A.off + m) : m;
  const long long mb = B.off ? (long long)__ldg(B.off + m) : m;
  const long long mo = out_off ? (long long)__ldg(out_off + m) : m;

  float2 acc[MG_TR][MG_TC];
#pragma unroll
  for (int r = 0; r < MG_TR; ++r)
#pragma unroll
    for (int c = 0; c < MG_TC; ++c) acc[r][c] = make_float2(0.f, 0.f);

  const float2* pa = A.ptr + ma;
  const float2* pb = B.ptr + mb;
#pragma unroll 2
  for (int k = 0; k < nK; ++k) {
    float2 a[MG_TR], b[MG_TC];
#pragma unroll
    for (int r = 0; r < MG_TR; ++r) {
      a[r] = (r0 + r < nR) ? __ldg(pa + (long long)(r0 + r) * A.s_outer + (long long)k * A.s_inner)
                           : make_float2(0.f, 0.f);
      if (CONJ_A) a[r].y = -a[r].y;
    }
#pragma unroll
    for (int c = 0; c < MG_TC; ++c) {
      b[c] = (c0 + c < nC) ? __ldg(pb + (long long)k * B.s_outer + (long long)(c0 + c) * B.s_inner)
                           : make_float2(0.f, 0.f);
      if (CONJ_B) b[c].y = -b[c].y;
    }
#pragma unroll
    for (int r = 0; r < MG_TR; ++r)
#pragma unroll
      for (int c = 0; c < MG_TC; ++c) {
        acc[r][c].x = fmaf(a[r].x, b[c].x, acc[r][c].x);
        acc[r][c].x = fmaf(-a[r].y, b[c].y, acc[r][c].x);
        acc[r][c].y = fmaf(a[r].x, b[c].y, acc[r][c].y);
        acc[r][c].y = fmaf(a[r].y, b[c].x, acc[r][c].y);
      }
  }
#pragma unroll
  for (int r = 0; r < MG_TR; ++r)
#pragma unroll
    for (int c = 0; c < MG_TC; ++c)
      if (r0 + r < nR && c0 + c < nC) outp[mo + (long long)(r0 + r) * so_r + (long long)(c0 + c) * so_c] = acc[r][c];
}

bool launch_mode_gemm(ModeGemmOperand A, bool conjA, ModeGemmOperand B, bool conjB, ModeGemmOperand Out, int nR,
                      int nC, int nK, int64_t nModes, cudaStream_t st) {
  if (nR <= 0 || nC <= 0 || nModes <= 0) return true;
  const int tiles = ((nR + MG_TR - 1) / MG_TR) * ((nC + MG_TC - 1) / MG_TC);
  dim3 grid((unsigned)((nModes + 31) / 32), (unsigned)((tiles + MG_WARPS - 1) / MG_WARPS));
  dim3 block(32, MG_WARPS);
  MgOp a{(const float2*)A.ptr, (long long)A.s_outer, (long long)A.s_inner, A.mode_off};
  MgOp b{(const float2*)B.ptr, (long long)B.s_outer, (long long)B.s_inner, B.mode_off};
  float2* o = (float2*)Out.ptr;
  if (conjA && !conjB)
    k_mode_gemm<true, false><<<grid, block, 0, st>>>(a, b, o, Out.s_outer, Out.s_inner, Out.mode_off, nR, nC, nK, nModes);
  else if (!conjA && conjB)
    k_mode_gemm<false, true><<<grid, block, 0, st>>>(a, b, o, Out.s_outer, Out.s_inner, Out.mode_off, nR, nC, nK, nModes);
  else if (!conjA && !conjB)
    k_mode_gemm<false, false><<<grid, block, 0, st>>>(a, b, o, Out.s_outer, Out.s_inner, Out.mode_off, nR, nC, nK, nModes);
  else
    k_mode_gemm<true, true><<<grid, block, 0, st>>>(a, b, o, Out.s_outer, Out.s_inner, Out.mode_off, nR, nC, nK, nModes);
  count_launch();
  return cuda_ok(cudaGetLastError(), "k_mode_gemm launch");
}

// =====================================================================================================
// 4. bias gradient from the DC slot of gm:  dbias[o] = inv_scale * sum_b Re(gm[b, o, dc])
// =====================================================================================================
__global__ void k_bias_grad(const float2* __restrict__ gm, float* __restrict__ dbias, int batch, int out_channels,
                            long long n_modes, int dc_slot, float inv_scale) {
  // one warp per output channel, lanes over the batch: the loads are independent (one L2 round trip), then a shuffle tree
  const int o = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (o >= out_channels) return;
  float s = 0.f;
  for (int b = lane; b < batch; b += 32) s += __ldg(&gm[((long long)b * out_channels + o) * n_modes + dc_slot].x);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
  if (lane == 0) dbias[o] = s * inv_scale;
}

bool launch_bias_grad(const float2* gm, float* dbias, int batch, int out_channels, int64_t n_modes, int dc_slot,
                      float inv_scale, cudaStream_t st) {
  if (out_channels <= 0) return true;
  k_bias_grad<<<(out_channels + 3) / 4, 128, 0, st>>>(gm, dbias, batch, out_channels, (long long)n_modes, dc_slot, inv_scale);
  count_launch();
  return cuda_ok(cudaGetLastError(), "k_bias_grad launch");
}

// =====================================================================================================
// 5. 16-bit image storage (SC_FLAG_GRID_F16 / SC_FLAG_GRID_BF16): x is widened to fp32 before the analysis, dx rounded to
//    nearest even after the adjoint synthesis.  Widening is exact, so the transforms see the very values the fp32 path would.
//    The element pair (sc_half.cuh) is shared with the tensor-core kernels and sc_hostcheck_convert.
// =====================================================================================================
constexpr int GC_THREADS = 256;
constexpr int GC_VEC = 8;   // elements per vector step: 16 bytes of 16-bit data, 32 bytes of float

// n_vec vector steps over 16-byte aligned buffers, then the scalar tail [8 n_vec, n)
template <int G, bool TO16>
__global__ void __launch_bounds__(GC_THREADS) k_grid_convert(const void* __restrict__ in, void* __restrict__ out, long long n,
                                                             long long n_vec) {
  const long long stride = (long long)gridDim.x * GC_THREADS;
  for (long long v = (long long)blockIdx.x * GC_THREADS + threadIdx.x; v < n_vec; v += stride) {
    if constexpr (TO16) {
      const float4* src = reinterpret_cast<const float4*>(in) + 2 * v;
      const float4 a = __ldg(src), b = __ldg(src + 1);
      const float f[GC_VEC] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
      uint32_t w[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) w[e] = (uint32_t)g16_store<G>(f[2 * e]) | ((uint32_t)g16_store<G>(f[2 * e + 1]) << 16);
      reinterpret_cast<uint4*>(out)[v] = make_uint4(w[0], w[1], w[2], w[3]);
    } else {
      const uint4 q = __ldg(reinterpret_cast<const uint4*>(in) + v);
      const uint32_t w[4] = {q.x, q.y, q.z, q.w};
      float f[GC_VEC];
#pragma unroll
      for (int e = 0; e < 4; ++e) { f[2 * e] = g16_load<G>((uint16_t)(w[e] & 0xffffu)); f[2 * e + 1] = g16_load<G>((uint16_t)(w[e] >> 16)); }
      float4* dst = reinterpret_cast<float4*>(out) + 2 * v;
      dst[0] = make_float4(f[0], f[1], f[2], f[3]);
      dst[1] = make_float4(f[4], f[5], f[6], f[7]);
    }
  }
  for (long long i = GC_VEC * n_vec + (long long)blockIdx.x * GC_THREADS + threadIdx.x; i < n; i += stride) {
    if constexpr (TO16) static_cast<uint16_t*>(out)[i] = g16_store<G>(static_cast<const float*>(in)[i]);
    else static_cast<float*>(out)[i] = g16_load<G>(static_cast<const uint16_t*>(in)[i]);
  }
}

bool launch_grid_convert(int grid16, const void* in, void* out, int64_t n, bool to_16, cudaStream_t st) {
  if (n <= 0) return true;
  if (grid16 != SC_FLAG_GRID_F16 && grid16 != SC_FLAG_GRID_BF16) { set_error("grid_convert: unknown 16-bit storage flag"); return false; }
  const bool aligned = ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 15u) == 0;
  const long long n_vec = aligned ? (long long)(n / GC_VEC) : 0;
  const long long work = n_vec > 0 ? n_vec : n;
  const unsigned blocks = (unsigned)std::min<long long>((work + GC_THREADS - 1) / GC_THREADS, 148LL * 16);
  if (grid16 == SC_FLAG_GRID_F16) {
    if (to_16) k_grid_convert<SC_FLAG_GRID_F16, true><<<blocks, GC_THREADS, 0, st>>>(in, out, (long long)n, n_vec);
    else k_grid_convert<SC_FLAG_GRID_F16, false><<<blocks, GC_THREADS, 0, st>>>(in, out, (long long)n, n_vec);
  } else {
    if (to_16) k_grid_convert<SC_FLAG_GRID_BF16, true><<<blocks, GC_THREADS, 0, st>>>(in, out, (long long)n, n_vec);
    else k_grid_convert<SC_FLAG_GRID_BF16, false><<<blocks, GC_THREADS, 0, st>>>(in, out, (long long)n, n_vec);
  }
  count_launch();
  return cuda_ok(cudaGetLastError(), "k_grid_convert launch");
}

}  // namespace sc

extern "C" int sc_hostcheck_convert(int flag, int to_16, const void* in, void* out, int64_t n) {
  using namespace sc;
  if ((flag != SC_FLAG_GRID_F16 && flag != SC_FLAG_GRID_BF16) || n < 0 || (n > 0 && (in == nullptr || out == nullptr))) {
    set_error("sc_hostcheck_convert: flag must be SC_FLAG_GRID_F16 or SC_FLAG_GRID_BF16, with n >= 0 elements");
    return 1;
  }
  for (int64_t i = 0; i < n; ++i) {
    if (to_16) {
      const float f = static_cast<const float*>(in)[i];
      static_cast<uint16_t*>(out)[i] = flag == SC_FLAG_GRID_F16 ? g16_store<SC_FLAG_GRID_F16>(f) : g16_store<SC_FLAG_GRID_BF16>(f);
    } else {
      const uint16_t b = static_cast<const uint16_t*>(in)[i];
      static_cast<float*>(out)[i] = flag == SC_FLAG_GRID_F16 ? g16_load<SC_FLAG_GRID_F16>(b) : g16_load<SC_FLAG_GRID_BF16>(b);
    }
  }
  return 0;
}
