// C ABI of libspectral_conv_b200.so: plan construction (kept-mode index set + twiddle tables) and the
// orchestration of the transform / contraction kernels.  See include/spectral_conv_b200.h for the contract
// and the reference lines each entry point replaces.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>

#include "sc_plan.h"
#include "sc_fast.h"

namespace sc {

static thread_local std::string t_error;
std::atomic<uint64_t> g_launches{0};

void set_error(const std::string& msg) { t_error = msg; }

bool cuda_ok(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return true;
  set_error(std::string(what) + ": " + cudaGetErrorString(e));
  return false;
}

template <typename T>
static bool upload(Plan* p, const std::vector<T>& host, T** dev) {
  if (p->host_only) { *dev = nullptr; return true; }   // table inspection without a device (sc_problem_table)
  void* d = nullptr;
  const size_t bytes = host.size() * sizeof(T);
  if (!cuda_ok(cudaMalloc(&d, bytes ? bytes : sizeof(T)), "cudaMalloc(table)")) return false;
  p->owned.push_back(d);
  if (bytes && !cuda_ok(cudaMemcpy(d, host.data(), bytes, cudaMemcpyHostToDevice), "cudaMemcpy(table)")) return false;
  *dev = static_cast<T*>(d);
  return true;
}

static const double kTwoPi = 6.283185307179586476925286766559;

// exp(sign * 2 pi i * (a*b mod n) / n) with the angle reduced in integers first
static inline void unit(long long a, long long b, long long n, int sign, double* re, double* im) {
  const long long r = ((a % n) * (b % n)) % n;
  const double ang = kTwoPi * (double)r / (double)n;
  *re = std::cos(ang);
  *im = sign * std::sin(ang);
}

// Kept-mode index set of one dim -- host only, no device state: what `SpectralConv.forward` derives at :465-519.
//   t->k        kept modes  min(F, n_modes)                                   (:466)
//   t->w0       first weight row used (`slices_w`)                            (:476-486)
//   t->in_bins  unshifted spectrum bin read by kept slot s (`slices_x` after undoing the fftshift of :449)   (:500-519)
static bool index_dim(const sc_problem& pr, int j, DimTables* tp) {
  DimTables& t = *tp;
  const bool last = (j == pr.ndim - 1);
  t.N = pr.grid[j];
  t.M = pr.out_grid[j];
  if (t.N < 1 || t.M < 1) { set_error("grid sizes must be >= 1"); return false; }
  if (pr.n_modes[j] < 1) { set_error("n_modes must be >= 1 along every dim"); return false; }
  t.F = last ? t.N / 2 + 1 : t.N;
  t.k = pr.n_modes[j] < t.F ? pr.n_modes[j] : t.F;                      // min(size, n_mode)   (:466)
  const int start = pr.max_n_modes[j] - t.k;                            // (:465-468)
  if (start < 0) { set_error("n_modes exceeds max_n_modes (weight too small for the requested modes)"); return false; }
  t.in_bins.resize(t.k);
  if (last) {
    t.w0 = 0;                                                           // slice(None, -start)  (:486)
    for (int s = 0; s < t.k; ++s) t.in_bins[s] = s;                      // slice(None, k)       (:514-517)
  } else {
    t.w0 = start ? start / 2 : 0;                                       // slice(start//2, -start//2) (:476-485)
    const int centre = t.F / 2, neg = t.k / 2;                          // (:507-512)
    for (int s = 0; s < t.k; ++s) {
      const int shifted = centre - neg + s;
      t.in_bins[s] = ((shifted - t.F / 2) % t.F + t.F) % t.F;           // undo fftshift = roll by F//2 (:449)
    }
  }
  // where each slot lands on the output grid
  t.out_bins.resize(t.k);
  for (int s = 0; s < t.k; ++s) {
    if (!last && (pr.flags & SC_FLAG_RESAMPLE)) {
      const int f = s - t.k / 2;                                        // signed frequency of the slot
      t.out_bins[s] = (t.k <= t.M) ? ((f % t.M) + t.M) % t.M : -1;     // resample.py:57-68
    } else {
      t.out_bins[s] = t.in_bins[s] < t.M ? t.in_bins[s] : -1;           // ifftn(s=M) crops / zero-pads the UNSHIFTED spectrum (:548)
    }
  }
  return true;
}

static bool build_plan(const sc_problem& pr, Plan* p) {
  p->prob = pr;
  p->d = pr.ndim;
  const int d = p->d;
  if (d < 1 || d > SC_MAX_DIMS) { set_error("ndim must be in 1..4"); return false; }
  if (pr.fft_norm < 0 || pr.fft_norm > 2) { set_error("unknown fft_norm"); return false; }
  if ((pr.flags & SC_FLAG_GRID_F16) && (pr.flags & SC_FLAG_GRID_BF16)) {
    set_error("SC_FLAG_GRID_F16 and SC_FLAG_GRID_BF16 exclude each other"); return false;
  }
  if ((pr.flags & (SC_FLAG_GRID_F16 | SC_FLAG_GRID_BF16)) && (pr.flags & SC_FLAG_RESAMPLE)) {
    set_error("16-bit image storage (SC_FLAG_GRID_F16 / SC_FLAG_GRID_BF16) is not available with SC_FLAG_RESAMPLE"); return false;
  }
  p->grid16 = pr.flags & (SC_FLAG_GRID_F16 | SC_FLAG_GRID_BF16);
  if (!p->host_only && !cuda_ok(cudaGetDevice(&p->device), "cudaGetDevice")) return false;

  p->n_modes_total = p->grid_points = p->out_points = p->weight_elems_per_io = 1;
  p->weight_block_is_whole = true;
  for (int j = 0; j < d; ++j) {
    DimTables& t = p->dim[j];
    if (!index_dim(pr, j, &t)) return false;
    const int start = pr.max_n_modes[j] - t.k;
    if (start != 0) p->weight_block_is_whole = false;
    p->n_modes_total *= t.k;
    p->grid_points *= t.N;
    p->out_points *= t.M;
    p->weight_elems_per_io *= pr.max_n_modes[j];
  }
  if (p->weight_elems_per_io * 1.0 > 2.0e9 || p->n_modes_total > (1ll << 30)) { set_error("mode block too large"); return false; }
  switch (pr.fft_norm) {
    case SC_NORM_FORWARD:  p->s_fwd = 1.0 / (double)p->grid_points; p->s_inv = 1.0; break;
    case SC_NORM_BACKWARD: p->s_fwd = 1.0; p->s_inv = 1.0 / (double)p->out_points; break;
    default: p->s_fwd = 1.0 / std::sqrt((double)p->grid_points); p->s_inv = 1.0 / std::sqrt((double)p->out_points);
  }

  // ---- leading dims: complex tables
  for (int j = 0; j + 1 < d; ++j) {
    DimTables& t = p->dim[j];
    std::vector<float2>&A = t.h_A, &AH = t.h_AH, &S = t.h_S, &SH = t.h_SH;
    A.assign((size_t)t.k * t.N, make_float2(0.f, 0.f));  AH.assign((size_t)t.N * t.k, make_float2(0.f, 0.f));
    S.assign((size_t)t.M * t.k, make_float2(0.f, 0.f));  SH.assign((size_t)t.k * t.M, make_float2(0.f, 0.f));
    for (int s = 0; s < t.k; ++s) {
      const int b = t.in_bins[s];
      for (int n = 0; n < t.N; ++n) {
        double re, im;
        unit(b, n, t.N, -1, &re, &im);
        A[(size_t)s * t.N + n] = make_float2((float)re, (float)im);
        AH[(size_t)n * t.k + s] = make_float2((float)re, (float)-im);
      }
      for (int n = 0; n < t.M; ++n) {
        double re = 0.0, im = 0.0;
        if (t.out_bins[s] >= 0) unit(t.out_bins[s], n, t.M, +1, &re, &im);
        S[(size_t)n * t.k + s] = make_float2((float)re, (float)im);
        SH[(size_t)s * t.M + n] = make_float2((float)re, (float)-im);
      }
    }
    if (!upload(p, A, &t.d_A) || !upload(p, AH, &t.d_AH) || !upload(p, S, &t.d_S) || !upload(p, SH, &t.d_SH)) return false;
  }
  // ---- last dim: real tables
  {
    DimTables& t = p->dim[d - 1];
    const int k2 = 2 * t.k;
    p->ldTA = k2; p->ldTAT = t.N; p->ldTS = t.M; p->ldTST = k2;
    std::vector<float>&TA = p->h_TA, &TAT = p->h_TAT, &TS = p->h_TS, &TST = p->h_TST;
    TA.assign((size_t)t.N * k2, 0.f);  TAT.assign((size_t)k2 * t.N, 0.f);
    TS.assign((size_t)k2 * t.M, 0.f);  TST.assign((size_t)t.M * k2, 0.f);
    for (int s = 0; s < t.k; ++s) {
      const int q = t.in_bins[s];
      for (int n = 0; n < t.N; ++n) {
        double re, im;
        unit(q, n, t.N, -1, &re, &im);
        const float c = (float)(p->s_fwd * re), sn = (float)(p->s_fwd * im);
        TA[(size_t)n * k2 + 2 * s] = c;      TA[(size_t)n * k2 + 2 * s + 1] = sn;
        TAT[(size_t)(2 * s) * t.N + n] = c;  TAT[(size_t)(2 * s + 1) * t.N + n] = sn;
      }
      // C2R rules: irfft(n=M) reads bins q < M/2+1; DC and (M even) Nyquist count once and ignore Im;
      // the reference also zeroes Im of the LAST bin of the input-sized spectrum when M is even (:552-559)
      const bool used = q < t.M / 2 + 1;
      const bool edge = (q == 0) || (t.M % 2 == 0 && q == t.M / 2);
      // (that zeroing of the last input bin is SpectralConv.forward's; `resample` hands the spectrum to irfftn untouched)
      const bool im_dead = edge || (!(pr.flags & SC_FLAG_RESAMPLE) && t.M % 2 == 0 && q == t.F - 1);
      const double cq = edge ? 1.0 : 2.0;
      for (int n = 0; n < t.M; ++n) {
        double re = 0.0, im = 0.0;
        if (used) unit(q, n, t.M, +1, &re, &im);
        const float c = (float)(p->s_inv * cq * re);
        const float sn = im_dead ? 0.f : (float)(-p->s_inv * cq * im);
        TS[(size_t)(2 * s) * t.M + n] = c;   TS[(size_t)(2 * s + 1) * t.M + n] = sn;
        TST[(size_t)n * k2 + 2 * s] = c;     TST[(size_t)n * k2 + 2 * s + 1] = sn;
      }
    }
    if (!upload(p, TA, &p->d_TA) || !upload(p, TAT, &p->d_TAT) || !upload(p, TS, &p->d_TS) || !upload(p, TST, &p->d_TST)) return false;
  }
  // ---- weight offsets of the kept block + DC slot
  {
    std::vector<int32_t> woff((size_t)p->n_modes_total);
    int64_t wstride[SC_MAX_DIMS];
    int64_t acc = 1;
    for (int j = d - 1; j >= 0; --j) { wstride[j] = acc; acc *= pr.max_n_modes[j]; }
    std::vector<int> idx(d, 0);
    for (int64_t m = 0; m < p->n_modes_total; ++m) {
      int64_t off = 0;
      for (int j = 0; j < d; ++j) off += (int64_t)(p->dim[j].w0 + idx[j]) * wstride[j];
      woff[(size_t)m] = (int32_t)off;
      for (int j = d - 1; j >= 0; --j) { if (++idx[j] < p->dim[j].k) break; idx[j] = 0; }
    }
    if (!upload(p, woff, &p->d_woff)) return false;
    int64_t dc = 0;
    for (int j = 0; j < d; ++j) dc = dc * p->dim[j].k + (j == d - 1 ? 0 : p->dim[j].k / 2);
    p->dc_slot = (int)dc;
  }
  return p->host_only ? true : fast_plan_init(p);
}

static inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

// largest intermediate of a transform chain over `n_images` images, in complex elements.  A chain state is
// "dims < s still on the grid (N for the forward pair, M for the adjoint pair), dims >= s already in mode space".
static int64_t chain_elems(const Plan* p, int64_t n_images) {
  const int d = p->d;
  int64_t best = 0;
  for (int variant = 0; variant < 2; ++variant) {
    for (int s = 1; s < d; ++s) {
      int64_t e = n_images;
      for (int j = 0; j < s; ++j) e *= variant ? p->dim[j].M : p->dim[j].N;
      for (int j = s; j < d; ++j) e *= p->dim[j].k;
      if (e > best) best = e;
    }
  }
  return best;
}

struct Workspace {
  float2* buf[2];
  float2* modes[2];
  float* grid32;     // 16-bit image storage only: the fp32 copy of x (analysis) or of dx (adjoint synthesis)
};

static size_t grid32_bytes(const Plan* p, int64_t n_images) {
  return p->grid16 ? align256((size_t)(n_images * p->grid_points) * sizeof(float)) : 0;
}

static bool carve(const Plan* p, int64_t n_images, void* ws, size_t ws_bytes, Workspace* out) {
  const size_t chain = align256((size_t)chain_elems(p, n_images) * sizeof(float2));
  const size_t modes = align256((size_t)(n_images * p->n_modes_total) * sizeof(float2));
  const size_t need = 2 * chain + 2 * modes + grid32_bytes(p, n_images);
  if (need > 0 && (ws == nullptr || ws_bytes < need)) { set_error("workspace too small (see sc_workspace_bytes)"); return false; }
  char* base = static_cast<char*>(ws);
  out->buf[0] = reinterpret_cast<float2*>(base);
  out->buf[1] = reinterpret_cast<float2*>(base + chain);
  out->modes[0] = reinterpret_cast<float2*>(base + 2 * chain);
  out->modes[1] = reinterpret_cast<float2*>(base + 2 * chain + modes);
  out->grid32 = p->grid16 ? reinterpret_cast<float*>(base + 2 * chain + 2 * modes) : nullptr;
  return true;
}

// ---- generic transform chains ---------------------------------------------------------------------------
static bool analyze_generic(const Plan* p, const float* images, int64_t n_images, float2* modes_out, bool adjoint,
                            float2* b0, float2* b1, cudaStream_t st) {
  const int d = p->d;
  const DimTables& L = p->dim[d - 1];
  int64_t lead = 1;
  for (int j = 0; j + 1 < d; ++j) lead *= adjoint ? p->dim[j].M : p->dim[j].N;
  const int64_t rows = n_images * lead;
  float2* cur = (d == 1) ? modes_out : b0;
  float2* nxt = b1;
  if (p->fast_enabled && rows_can_analyze(p, adjoint, rows) &&
      ((reinterpret_cast<uintptr_t>(images) | reinterpret_cast<uintptr_t>(cur)) & 15u) == 0) {
    if (!rows_analyze(p, images, rows, reinterpret_cast<float*>(cur), adjoint, st)) return false;
  } else
  if (!launch_real_table_gemm(images, adjoint ? p->d_TST : p->d_TA, adjoint ? p->ldTST : p->ldTA,
                              reinterpret_cast<float*>(cur), nullptr, rows, adjoint ? L.M : L.N, 2 * L.k, 1, 1, st))
    return false;
  int64_t inner = L.k;
  for (int j = d - 2; j >= 0; --j) {
    const DimTables& t = p->dim[j];
    const int Q = adjoint ? t.M : t.N;
    lead /= Q;
    float2* dst = (j == 0) ? modes_out : nxt;
    if (!launch_complex_table_gemm(adjoint ? t.d_SH : t.d_A, cur, dst, n_images * lead, t.k, Q, (int)inner, st)) return false;
    inner *= t.k;
    nxt = cur; cur = dst;
  }
  return true;
}

static bool synthesize_generic(const Plan* p, const float2* modes_in, int64_t n_images, int n_channels,
                               const float* bias, float* images_out, bool adjoint, float2* b0, float2* b1,
                               cudaStream_t st) {
  const int d = p->d;
  const DimTables& L = p->dim[d - 1];
  const float2* cur = modes_in;
  float2* bufs[2] = {b0, b1};
  int which = 0;
  int64_t lead = 1;
  int64_t inner = p->n_modes_total;
  for (int j = 0; j + 1 < d; ++j) {
    const DimTables& t = p->dim[j];
    const int P = adjoint ? t.N : t.M;
    inner /= t.k;
    float2* dst = bufs[which];
    if (!launch_complex_table_gemm(adjoint ? t.d_AH : t.d_S, cur, dst, n_images * lead, P, t.k, (int)inner, st)) return false;
    lead *= P;
    cur = dst; which ^= 1;
  }
  const int64_t rows = n_images * lead;
  if (p->fast_enabled && rows_can_synthesize(p, adjoint, rows) &&
      ((reinterpret_cast<uintptr_t>(images_out) | reinterpret_cast<uintptr_t>(cur)) & 15u) == 0)
    return rows_synthesize(p, reinterpret_cast<const float*>(cur), rows, images_out, bias, lead, n_channels > 0 ? n_channels : 1,
                           adjoint, st);
  return launch_real_table_gemm(reinterpret_cast<const float*>(cur), adjoint ? p->d_TAT : p->d_TS,
                                adjoint ? p->ldTAT : p->ldTS, images_out, bias, rows, 2 * L.k, adjoint ? L.N : L.M,
                                lead, n_channels > 0 ? n_channels : 1, st);
}

static bool analyze32(const Plan* p, const float* images, int64_t n_images, float2* modes_out, bool adjoint,
                      float2* b0, float2* b1, cudaStream_t st, bool quad_major, const L2Prefetch* pf, int storage) {
  if (n_images <= 0) return true;
  if (quad_major) return fast_analyze(p, images, n_images, modes_out, adjoint, st, true, pf, storage);   // (dense_chain_quad_major checked the shape)
  // tensor maps and bulk copies need 16-byte aligned bases: an offset view (e.g. buf[1:].view(...)) takes the generic chain
  const bool aligned = ((reinterpret_cast<uintptr_t>(images) | reinterpret_cast<uintptr_t>(modes_out)) & 15u) == 0;
  if (p->fast_enabled && aligned && fast_can_analyze(p, adjoint)) {
    if (p->d == 2) {
      if (n_images % fast_tile_group(p, false, adjoint) == 0)
        return fast_analyze(p, images, n_images, modes_out, adjoint, st, false, pf, storage);
    } else {   // d == 3: fused last two dims per (image, z) slice, then dim 0 on the truncated data
      const DimTables& Z = p->dim[0];
      const int64_t slices = n_images * (adjoint ? Z.M : Z.N);
      if (slices % fast_tile_group(p, false, adjoint) == 0) {
        if (!fast_analyze(p, images, slices, b0, adjoint, st, false, nullptr, storage)) return false;
        const int64_t inner = (int64_t)p->dim[1].k * p->dim[2].k;
        return launch_complex_table_gemm(adjoint ? Z.d_SH : Z.d_A, b0, modes_out, n_images, Z.k, adjoint ? Z.M : Z.N, (int)inner, st);
      }
    }
  }
  if (storage != 0) { set_error("analyze: 16-bit images reached the float-only chain"); return false; }
  return analyze_generic(p, images, n_images, modes_out, adjoint, b0, b1, st);
}

static bool synthesize32(const Plan* p, const float2* modes_in, int64_t n_images, int n_channels, const float* bias,
                         float* images_out, bool adjoint, float2* b0, float2* b1, cudaStream_t st, bool quad_major, int storage) {
  if (n_images <= 0) return true;
  if (quad_major) return fast_synthesize(p, modes_in, n_images, n_channels, bias, images_out, adjoint, 1, st, true, storage);
  const bool aligned = ((reinterpret_cast<uintptr_t>(images_out) | reinterpret_cast<uintptr_t>(modes_in)) & 15u) == 0;
  if (p->fast_enabled && aligned && fast_can_synthesize(p, adjoint)) {
    if (p->d == 2) {
      if (n_images % fast_tile_group(p, true, adjoint) == 0)
        return fast_synthesize(p, modes_in, n_images, n_channels, bias, images_out, adjoint, 1, st, false, storage);
    } else {
      const DimTables& Z = p->dim[0];
      const int P0 = adjoint ? Z.N : Z.M;
      const int64_t slices = n_images * P0;
      if (slices % fast_tile_group(p, true, adjoint) == 0) {
        const int64_t inner = (int64_t)p->dim[1].k * p->dim[2].k;
        if (!launch_complex_table_gemm(adjoint ? Z.d_AH : Z.d_S, modes_in, b0, n_images, P0, Z.k, (int)inner, st)) return false;
        return fast_synthesize(p, b0, slices, n_channels, bias, images_out, adjoint, P0, st, false, storage);
      }
    }
  }
  if (storage != 0) { set_error("synthesize: 16-bit images reached the float-only chain"); return false; }
  return synthesize_generic(p, modes_in, n_images, n_channels, bias, images_out, adjoint, b0, b1, st);
}

// Whether analyze32 / synthesize32 take the fused tensor-core kernels for this call (the same tests they make, in the same order).
static bool fused_analysis_taken(const Plan* p, const void* images, int64_t n_images, const void* modes_out, bool adjoint, bool quad_major) {
  if (quad_major) return true;
  const bool aligned = ((reinterpret_cast<uintptr_t>(images) | reinterpret_cast<uintptr_t>(modes_out)) & 15u) == 0;
  if (!(p->fast_enabled && aligned && fast_can_analyze(p, adjoint))) return false;
  const int64_t units = p->d == 2 ? n_images : n_images * (adjoint ? p->dim[0].M : p->dim[0].N);
  return (p->d == 2 || p->d == 3) && units % fast_tile_group(p, false, adjoint) == 0;
}

static bool fused_synthesis_taken(const Plan* p, const void* modes_in, int64_t n_images, const void* images_out, bool adjoint, bool quad_major) {
  if (quad_major) return true;
  const bool aligned = ((reinterpret_cast<uintptr_t>(images_out) | reinterpret_cast<uintptr_t>(modes_in)) & 15u) == 0;
  if (!(p->fast_enabled && aligned && fast_can_synthesize(p, adjoint))) return false;
  const int64_t units = p->d == 2 ? n_images : n_images * (adjoint ? p->dim[0].N : p->dim[0].M);
  return (p->d == 2 || p->d == 3) && units % fast_tile_group(p, true, adjoint) == 0;
}

// The storage type of the images on `grid` is decided here and nowhere else.  With 16-bit storage the fused tensor-core kernels
// read x / write dx at 16 bits themselves (k_fused_analysis2 widens each element before its hi / lo split, k_fused_synthesis
// rounds in its epilogue); every other chain -- a misaligned view, the rows and generic kernels, the first-generation analysis --
// runs on an fp32 copy in the workspace (widened exactly before the analysis, rounded to nearest even after the adjoint synthesis).
// Either way the arithmetic is that of the float path on the widened input.  y / gy are always float.
static bool analyze(const Plan* p, const float* images, int64_t n_images, float2* modes_out, bool adjoint, const Workspace& w,
                    cudaStream_t st, bool quad_major = false, const L2Prefetch* pf = nullptr) {
  if (n_images <= 0) return true;
  if (p->grid16 && !adjoint) {
    if (((reinterpret_cast<uintptr_t>(images) & 15u) == 0) && fast_analysis_reads_16bit(p) &&
        fused_analysis_taken(p, images, n_images, modes_out, adjoint, quad_major))
      return analyze32(p, images, n_images, modes_out, adjoint, w.buf[0], w.buf[1], st, quad_major, pf, p->grid16);
    if (!launch_grid_convert(p->grid16, images, w.grid32, n_images * p->grid_points, false, st)) return false;
    images = w.grid32;
  }
  return analyze32(p, images, n_images, modes_out, adjoint, w.buf[0], w.buf[1], st, quad_major, pf, 0);
}

static bool synthesize(const Plan* p, const float2* modes_in, int64_t n_images, int n_channels, const float* bias,
                       float* images_out, bool adjoint, const Workspace& w, cudaStream_t st, bool quad_major = false) {
  if (n_images <= 0) return true;
  if (p->grid16 && adjoint) {
    if (((reinterpret_cast<uintptr_t>(images_out) & 15u) == 0) && fused_synthesis_taken(p, modes_in, n_images, images_out, adjoint, quad_major))
      return synthesize32(p, modes_in, n_images, n_channels, bias, images_out, adjoint, w.buf[0], w.buf[1], st, quad_major, p->grid16);
    return synthesize32(p, modes_in, n_images, n_channels, bias, w.grid32, adjoint, w.buf[0], w.buf[1], st, quad_major, 0) &&
           launch_grid_convert(p->grid16, w.grid32, images_out, n_images * p->grid_points, true, st);
  }
  return synthesize32(p, modes_in, n_images, n_channels, bias, images_out, adjoint, w.buf[0], w.buf[1], st, quad_major, 0);
}

// `chained`: the call is part of sc_forward_dense / sc_backward_dense, i.e. the kernel launched just before on the stream is
// this library's transform kernel, which does not write the weights / saved modes: the contraction may fetch those operands
// ahead of its grid-dependency wait.  Standalone calls (chained = false) make no assumption about their predecessor.
//
// Quad-major mode tensors (x_qm / y_qm / g_qm): inside the dense chains the kept-mode tensors are internal, so they are
// laid out [quad of 4 modes][batch][channel][4] instead of [batch][channel][modes]: the 32-byte sectors one contraction CTA
// touches are then contiguous along the channel index and its loads / stores coalesce (the standard layout costs one L1
// wavefront per sector: measured LSU-bound).  Only the strides of the launch change.
static bool l2_resident_env() {   // SC_CONTRACT_PREFETCH=1: keep the contraction's own L2 prefetches inside the chains too (A/B runs)
  static const bool v = [] { const char* e = getenv("SC_CONTRACT_PREFETCH"); return e == nullptr || atoi(e) == 0; }();
  return v;
}

static bool contract_fwd(const Plan* p, const float2* xm, const float2* w, float2* ym, int B, int Ci, int Co,
                         cudaStream_t st, bool chained, bool x_qm = false, bool y_qm = false) {
  const int64_t Mt = p->n_modes_total, Wp = p->weight_elems_per_io;
  const bool quad_ok = mode_gemm_quad_eligible(p, Mt, w, xm, ym);
  if ((x_qm || y_qm) && !(quad_ok && quad2_enabled())) { set_error("quad-major mode tensors need the quad contraction kernel"); return false; }
  if ((p->fast_enabled || x_qm || y_qm) && fast_can_contract(p, B, Ci, Co, quad_ok)) {   // ym^T[o, b] = sum_i w[i, o] * xm[b, i]
    ModeGemmExtras ex;
    ex.a_early = chained;
    ex.l2_resident = chained && l2_resident_env();
    long long sBN = (long long)Ci * Mt, sBK = Mt, sOR = Mt, sON = (long long)Co * Mt;
    if (x_qm) { ex.sBQ = (long long)B * Ci * 4; sBN = (long long)Ci * 4; sBK = 4; }
    if (y_qm) { ex.sOQ = (long long)B * Co * 4; sOR = 4; sON = (long long)Co * 4; }
    return launch_mode_gemm_tc(p, w, Wp, (long long)Co * Wp, p->d_woff, false, xm, sBN, sBK, nullptr, ym, sOR, sON, nullptr, Co, B,
                               Ci, Mt, st, &ex);
  }
  ModeGemmOperand a{xm, (int64_t)Ci * Mt, Mt, nullptr};
  ModeGemmOperand b{w, (int64_t)Co * Wp, Wp, p->d_woff};
  ModeGemmOperand o{ym, (int64_t)Co * Mt, Mt, nullptr};
  return launch_mode_gemm(a, false, b, false, o, B, Co, Ci, Mt, st);
}

static bool contract_bwd(const Plan* p, const float2* xm, const float2* gm, const float2* w, float2* dxm,
                         float2* dw, float* dbias, int B, int Ci, int Co, cudaStream_t st, bool chained,
                         bool x_qm = false, bool g_qm = false, cudaEvent_t grads_ready = nullptr) {
  const int64_t Mt = p->n_modes_total, Wp = p->weight_elems_per_io;
  const bool quad_ok = (dw == nullptr || mode_gemm_quad_eligible(p, Mt, xm, gm, dw)) &&
                       (dxm == nullptr || mode_gemm_quad_eligible(p, Mt, w, gm, dxm));
  const bool any_qm = (x_qm && dw != nullptr) || g_qm;
  if (any_qm && !(quad_ok && quad2_enabled())) { set_error("quad-major mode tensors need the quad contraction kernel (32-byte aligned operands)"); return false; }
  const bool tc = (p->fast_enabled || any_qm) && fast_can_contract(p, B, Ci, Co, quad_ok);
  if (dw != nullptr && !p->weight_block_is_whole &&
      !cuda_ok(cudaMemsetAsync(dw, 0, (size_t)Ci * Co * Wp * sizeof(float2), st), "cudaMemsetAsync(dweight)"))
    return false;
  if (tc) {
    bool bias_done = false, have_dw_launch = false;
    // gm as an operand: rows o / k = b (dweight) or rows b / k = o (dxm)
    const long long g_sB = g_qm ? (long long)Co * 4 : (long long)Co * Mt, g_sO = g_qm ? 4 : Mt, g_sQ = g_qm ? (long long)B * Co * 4 : 0;
    // dweight[i, o] = sum_b conj(xm[b, i]) * gm[b, o]   (+ dbias from the DC slot of gm, fused into the same launch)
    if (dw != nullptr) {
      ModeGemmExtras ex;
      ex.a_early = chained;                          // the saved modes come from the forward pass
      ex.l2_resident = chained && l2_resident_env();
      if (dbias != nullptr) { ex.dbias = dbias; ex.bias_scale = (float)(1.0 / p->s_inv); }
      long long sAR = Mt, sAK = (long long)Ci * Mt;
      if (x_qm) { ex.sAQ = (long long)B * Ci * 4; sAR = 4; sAK = (long long)Ci * 4; }
      ex.sBQ = g_sQ;
      if (!launch_mode_gemm_tc(p, xm, sAR, sAK, nullptr, true, gm, g_sO, g_sB, nullptr, dw,
                               (long long)Co * Wp, Wp, p->d_woff, Ci, Co, B, Mt, st, &ex))
        return false;
      bias_done = ex.bias_done;
      have_dw_launch = true;
    }
    if (dbias != nullptr && !bias_done) {
      if (g_qm) { set_error("bias gradient from a quad-major gm needs the dweight launch"); return false; }
      if (!launch_bias_grad(gm, dbias, B, Co, Mt, p->dc_slot, (float)(1.0 / p->s_inv), st)) return false;
    }
    // dweight and dbias are complete once the launches above retire: a data-parallel caller starts its gradient all-reduce
    // on this event, underneath the dxm product and the dx synthesis
    if (grads_ready != nullptr && !cuda_ok(cudaEventRecord(grads_ready, st), "cudaEventRecord(grads_ready)")) return false;
    // dxm^T[i, b] = sum_o conj(w[i, o]) * gm[b, o]
    if (dxm != nullptr) {
      ModeGemmExtras ex;
      // the kernel just before this one is the dweight / bias-gradient launch above (when there was one), which writes
      // neither the weights nor gm
      ex.a_early = chained || have_dw_launch;
      ex.b_early = have_dw_launch;
      ex.l2_resident = chained && l2_resident_env();
      ex.sBQ = g_sQ;
      long long sOR = Mt, sON = (long long)Ci * Mt;
      if (g_qm) { ex.sOQ = (long long)B * Ci * 4; sOR = 4; sON = (long long)Ci * 4; }
      if (!launch_mode_gemm_tc(p, w, (long long)Co * Wp, Wp, p->d_woff, true, gm, g_sB, g_sO, nullptr, dxm, sOR, sON, nullptr,
                               Ci, B, Co, Mt, st, &ex))
        return false;
    }
    return true;
  }
  if (dw != nullptr) {
    ModeGemmOperand a{xm, Mt, (int64_t)Ci * Mt, nullptr};          // r = i, k = b
    ModeGemmOperand b{gm, (int64_t)Co * Mt, Mt, nullptr};          // k = b, c = o
    ModeGemmOperand o{dw, (int64_t)Co * Wp, Wp, p->d_woff};
    if (!launch_mode_gemm(a, true, b, false, o, Ci, Co, B, Mt, st)) return false;
  }
  if (dbias != nullptr &&
      !launch_bias_grad(gm, dbias, B, Co, Mt, p->dc_slot, (float)(1.0 / p->s_inv), st))
    return false;
  if (grads_ready != nullptr && !cuda_ok(cudaEventRecord(grads_ready, st), "cudaEventRecord(grads_ready)")) return false;
  if (dxm != nullptr) {
    ModeGemmOperand a{gm, (int64_t)Co * Mt, Mt, nullptr};          // r = b, k = o
    ModeGemmOperand b{w, Wp, (int64_t)Co * Wp, p->d_woff};         // k = o, c = i  (conjugated)
    ModeGemmOperand o{dxm, (int64_t)Ci * Mt, Mt, nullptr};
    if (!launch_mode_gemm(a, false, b, true, o, B, Ci, Co, Mt, st)) return false;
  }
  return true;
}

// The dense chains keep their mode tensors quad-major when every stage is a kernel that speaks that layout: 2-D problem on
// the fused tcgen05 transforms (whole tiles), quad contraction (whole weight block, mode count a multiple of 4, aligned weight).
static bool dense_chain_quad_major(const Plan* p, int B, int Ci, int Co, const void* weight) {
  static const bool env_on = [] { const char* e = getenv("SC_QUAD_MAJOR"); return e == nullptr || atoi(e) != 0; }();   // =0: A/B runs
  if (!env_on || !p->fast_enabled || p->fast == nullptr || p->d != 2 || !quad2_enabled()) return false;
  if (!fast_can_analyze(p, false) || !fast_can_analyze(p, true) || !fast_can_synthesize(p, false) || !fast_can_synthesize(p, true)) return false;
  const int64_t ni = (int64_t)B * Ci, no = (int64_t)B * Co;
  if (ni % fast_tile_group(p, false, false) || no % fast_tile_group(p, true, false) || no % fast_tile_group(p, false, true) ||
      ni % fast_tile_group(p, true, true))
    return false;
  return p->weight_block_is_whole && p->n_modes_total % 4 == 0 && (reinterpret_cast<uintptr_t>(weight) & 31u) == 0;
}

}  // namespace sc

using namespace sc;

#define SC_TRY(expr) do { if (!(expr)) return 1; } while (0)
#define SC_REQUIRE(cond, msg) do { if (!(cond)) { set_error(msg); return 1; } } while (0)

extern "C" {

int sc_plan_create(const sc_problem* problem, sc_plan** plan_out) {
  SC_REQUIRE(problem != nullptr && plan_out != nullptr, "sc_plan_create: null argument");
  Plan* p = new (std::nothrow) Plan();
  SC_REQUIRE(p != nullptr, "sc_plan_create: out of host memory");
  if (!build_plan(*problem, p)) {
    for (void* d : p->owned) cudaFree(d);
    delete p;
    return 1;
  }
  *plan_out = reinterpret_cast<sc_plan*>(p);
  return 0;
}

void sc_plan_destroy(sc_plan* plan) {
  if (plan == nullptr) return;
  Plan* p = reinterpret_cast<Plan*>(plan);
  fast_plan_destroy(p);
  for (void* d : p->owned) cudaFree(d);
  delete p;
}

int sc_plan_kept_modes(const sc_plan* plan, int32_t* kept_out) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  if (p == nullptr || kept_out == nullptr) return 0;
  for (int j = 0; j < p->d; ++j) kept_out[j] = p->dim[j].k;
  return p->d;
}

int sc_problem_table(const sc_problem* problem, int which, int dim, float* out, size_t out_capacity_floats,
                     int64_t* rows_out, int64_t* cols_out) {
  SC_REQUIRE(problem != nullptr && rows_out != nullptr && cols_out != nullptr, "sc_problem_table: null argument");
  Plan plan;
  plan.host_only = true;
  SC_TRY(build_plan(*problem, &plan));
  const int d = plan.d;
  const float* src = nullptr;
  int64_t rows = 0, cols = 0;       // cols counts floats (complex tables: 2 per entry)
  const DimTables& last = plan.dim[d - 1];
  switch (which) {
    case SC_TABLE_LAST_ANALYSIS:          src = plan.h_TA.data();  rows = last.N;     cols = 2 * last.k; break;
    case SC_TABLE_LAST_ANALYSIS_ADJOINT:  src = plan.h_TAT.data(); rows = 2 * last.k; cols = last.N;     break;
    case SC_TABLE_LAST_SYNTHESIS:         src = plan.h_TS.data();  rows = 2 * last.k; cols = last.M;     break;
    case SC_TABLE_LAST_SYNTHESIS_ADJOINT: src = plan.h_TST.data(); rows = last.M;     cols = 2 * last.k; break;
    default: {
      SC_REQUIRE(dim >= 0 && dim < d - 1, "sc_problem_table: leading-dim tables need 0 <= dim < ndim - 1");
      const DimTables& t = plan.dim[dim];
      switch (which) {
        case SC_TABLE_LEAD_ANALYSIS:          src = &t.h_A[0].x;  rows = t.k; cols = 2 * (int64_t)t.N; break;
        case SC_TABLE_LEAD_ANALYSIS_ADJOINT:  src = &t.h_AH[0].x; rows = t.N; cols = 2 * (int64_t)t.k; break;
        case SC_TABLE_LEAD_SYNTHESIS:         src = &t.h_S[0].x;  rows = t.M; cols = 2 * (int64_t)t.k; break;
        case SC_TABLE_LEAD_SYNTHESIS_ADJOINT: src = &t.h_SH[0].x; rows = t.k; cols = 2 * (int64_t)t.M; break;
        default: SC_REQUIRE(false, "sc_problem_table: unknown table id");
      }
    }
  }
  *rows_out = rows;
  *cols_out = cols;
  if (out != nullptr) {
    SC_REQUIRE((size_t)(rows * cols) <= out_capacity_floats, "sc_problem_table: output buffer too small");
    memcpy(out, src, (size_t)(rows * cols) * sizeof(float));
  }
  return 0;
}

int sc_problem_mode_bins(const sc_problem* problem, int dim, int32_t* kept_out, int32_t* in_bins_out,
                         int32_t* weight_rows_out) {
  SC_REQUIRE(problem != nullptr && problem->ndim >= 1 && problem->ndim <= SC_MAX_DIMS && dim >= 0 && dim < problem->ndim,
             "sc_problem_mode_bins: bad argument");
  DimTables t;
  SC_TRY(index_dim(*problem, dim, &t));
  if (kept_out) *kept_out = t.k;
  for (int s = 0; s < t.k; ++s) {
    if (in_bins_out) in_bins_out[s] = t.in_bins[s];
    if (weight_rows_out) weight_rows_out[s] = t.w0 + s;
  }
  return 0;
}

int sc_plan_mode_bins(const sc_plan* plan, int dim, int32_t* in_bins_out, int32_t* weight_rows_out) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  SC_REQUIRE(p != nullptr && dim >= 0 && dim < p->d, "sc_plan_mode_bins: bad argument");
  for (int s = 0; s < p->dim[dim].k; ++s) {
    if (in_bins_out) in_bins_out[s] = p->dim[dim].in_bins[s];
    if (weight_rows_out) weight_rows_out[s] = p->dim[dim].w0 + s;
  }
  return 0;
}

size_t sc_workspace_bytes(const sc_plan* plan, int64_t n_images) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  if (p == nullptr || n_images <= 0) return 0;
  return 2 * align256((size_t)chain_elems(p, n_images) * sizeof(float2)) +
         2 * align256((size_t)(n_images * p->n_modes_total) * sizeof(float2)) + grid32_bytes(p, n_images);
}

int sc_plan_set_fast_path(sc_plan* plan, int enable) {
  SC_REQUIRE(plan != nullptr, "sc_plan_set_fast_path: null plan");
  reinterpret_cast<Plan*>(plan)->fast_enabled = enable != 0;
  return 0;
}

int sc_plan_set_reserved_sms(sc_plan* plan, int n_sms) {
  SC_REQUIRE(plan != nullptr && n_sms >= 0, "sc_plan_set_reserved_sms: bad argument");
  reinterpret_cast<Plan*>(plan)->reserved_sms = n_sms;
  return 0;
}

int sc_plan_uses_fast_path(const sc_plan* plan) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  if (p == nullptr || !p->fast_enabled) return 0;
  int mask = (fast_can_analyze(p, false) ? 1 : 0) | (fast_can_synthesize(p, false) ? 2 : 0) |
             (fast_can_analyze(p, true) ? 4 : 0) | (fast_can_synthesize(p, true) ? 8 : 0);
  // bits 4-7: the last-dim ("rows") tensor-core kernels are available for the generic chain (row count permitting)
  mask |= (rows_can_analyze(p, false, 128) ? 16 : 0) | (rows_can_synthesize(p, false, 128) ? 32 : 0) |
          (rows_can_analyze(p, true, 128) ? 64 : 0) | (rows_can_synthesize(p, true, 128) ? 128 : 0);
  return mask;
}

int sc_analyze(const sc_plan* plan, const float* images, int64_t n_images, sc_complex* modes_out, int adjoint,
               void* workspace, size_t workspace_bytes, sc_stream stream) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  SC_REQUIRE(p != nullptr && images != nullptr && modes_out != nullptr, "sc_analyze: null argument");
  Workspace w{};
  SC_TRY(carve(p, n_images, workspace, workspace_bytes, &w));
  SC_TRY(analyze(p, images, n_images, reinterpret_cast<float2*>(modes_out), adjoint != 0, w, static_cast<cudaStream_t>(stream)));
  return 0;
}

int sc_synthesize(const sc_plan* plan, const sc_complex* modes_in, int64_t n_images, int32_t n_channels,
                  const float* bias, float* images_out, int adjoint, void* workspace, size_t workspace_bytes,
                  sc_stream stream) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  SC_REQUIRE(p != nullptr && modes_in != nullptr && images_out != nullptr, "sc_synthesize: null argument");
  SC_REQUIRE(!(adjoint && bias != nullptr), "sc_synthesize: bias is only valid for the forward synthesis");
  SC_REQUIRE(bias == nullptr || n_channels > 0, "sc_synthesize: n_channels must be > 0 with a bias");
  Workspace w{};
  SC_TRY(carve(p, n_images, workspace, workspace_bytes, &w));
  SC_TRY(synthesize(p, reinterpret_cast<const float2*>(modes_in), n_images, n_channels, bias, images_out,
                    adjoint != 0, w, static_cast<cudaStream_t>(stream)));
  return 0;
}

int sc_contract_dense(const sc_plan* plan, const sc_complex* xm, const sc_complex* weight, sc_complex* ym,
                      int32_t batch, int32_t in_channels, int32_t out_channels, sc_stream stream) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  SC_REQUIRE(p != nullptr && xm != nullptr && weight != nullptr && ym != nullptr, "sc_contract_dense: null argument");
  SC_TRY(contract_fwd(p, reinterpret_cast<const float2*>(xm), reinterpret_cast<const float2*>(weight),
                      reinterpret_cast<float2*>(ym), batch, in_channels, out_channels, static_cast<cudaStream_t>(stream), false));
  return 0;
}

int sc_contract_dense_backward(const sc_plan* plan, const sc_complex* xm, const sc_complex* gm,
                               const sc_complex* weight, sc_complex* dxm, sc_complex* dweight, float* dbias,
                               int32_t batch, int32_t in_channels, int32_t out_channels, sc_stream stream) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  SC_REQUIRE(p != nullptr && gm != nullptr, "sc_contract_dense_backward: null argument");
  SC_REQUIRE(dweight == nullptr || xm != nullptr, "sc_contract_dense_backward: dweight needs xm");
  SC_REQUIRE(dxm == nullptr || weight != nullptr, "sc_contract_dense_backward: dxm needs weight");
  SC_TRY(contract_bwd(p, reinterpret_cast<const float2*>(xm), reinterpret_cast<const float2*>(gm),
                      reinterpret_cast<const float2*>(weight), reinterpret_cast<float2*>(dxm),
                      reinterpret_cast<float2*>(dweight), dbias, batch, in_channels, out_channels,
                      static_cast<cudaStream_t>(stream), false));
  return 0;
}

int sc_bias_grad(const sc_plan* plan, const sc_complex* gm, float* dbias, int32_t batch, int32_t out_channels,
                 sc_stream stream) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  SC_REQUIRE(p != nullptr && gm != nullptr && dbias != nullptr, "sc_bias_grad: null argument");
  SC_TRY(launch_bias_grad(reinterpret_cast<const float2*>(gm), dbias, batch, out_channels, p->n_modes_total,
                          p->dc_slot, (float)(1.0 / p->s_inv), static_cast<cudaStream_t>(stream)));
  return 0;
}

int sc_forward_dense(const sc_plan* plan, const float* x, const sc_complex* weight, const float* bias, float* y,
                     sc_complex* xm_saved, int32_t* saved_layout_out, int32_t batch, int32_t in_channels, int32_t out_channels,
                     void* workspace, size_t workspace_bytes, sc_stream stream) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  SC_REQUIRE(p != nullptr && x != nullptr && weight != nullptr && y != nullptr && xm_saved != nullptr,
             "sc_forward_dense: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t n_max = (int64_t)batch * (in_channels > out_channels ? in_channels : out_channels);
  Workspace w{};
  SC_TRY(carve(p, n_max, workspace, workspace_bytes, &w));
  float2* xm = reinterpret_cast<float2*>(xm_saved);
  float2* ym = w.modes[0];
  // without a place to report it the saved modes stay in the standard layout
  const bool qm = saved_layout_out != nullptr && dense_chain_quad_major(p, batch, in_channels, out_channels, weight) &&
                  (reinterpret_cast<uintptr_t>(xm_saved) & 31u) == 0 &&
                  (((p->grid16 ? 0 : reinterpret_cast<uintptr_t>(x)) | reinterpret_cast<uintptr_t>(y)) & 15u) == 0;   // 16-bit x: read from the workspace copy
  if (saved_layout_out != nullptr) *saved_layout_out = qm ? SC_MODES_QUAD_MAJOR : SC_MODES_STANDARD;
  // the forward contraction reads the whole weight right after the analysis: let the analysis launch pull it into L2
  L2Prefetch pf;
  pf.ptr[0] = weight; pf.bytes[0] = (unsigned long long)in_channels * out_channels * p->weight_elems_per_io * sizeof(float2);
  SC_TRY(analyze(p, x, (int64_t)batch * in_channels, xm, false, w, st, qm, &pf));
  SC_TRY(contract_fwd(p, xm, reinterpret_cast<const float2*>(weight), ym, batch, in_channels, out_channels, st, true, qm, qm));
  SC_TRY(synthesize(p, ym, (int64_t)batch * out_channels, out_channels, bias, y, false, w, st, qm));
  return 0;
}

int sc_backward_dense(const sc_plan* plan, const float* gy, const sc_complex* weight, const sc_complex* xm_saved,
                      int32_t saved_layout, float* dx, sc_complex* dweight, float* dbias, int32_t batch, int32_t in_channels,
                      int32_t out_channels, void* workspace, size_t workspace_bytes, sc_stream stream, sc_event grads_ready) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  SC_REQUIRE(p != nullptr && gy != nullptr && weight != nullptr, "sc_backward_dense: null argument");
  SC_REQUIRE(dweight == nullptr || xm_saved != nullptr, "sc_backward_dense: dweight needs the saved modes");
  SC_REQUIRE(saved_layout == SC_MODES_STANDARD || saved_layout == SC_MODES_QUAD_MAJOR, "sc_backward_dense: unknown saved_layout");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t n_max = (int64_t)batch * (in_channels > out_channels ? in_channels : out_channels);
  Workspace w{};
  SC_TRY(carve(p, n_max, workspace, workspace_bytes, &w));
  float2* gm = w.modes[0];
  float2* dxm = dx != nullptr ? w.modes[1] : nullptr;
  const bool x_qm = saved_layout == SC_MODES_QUAD_MAJOR;
  // gm / dxm are internal to this call: quad-major whenever the chain allows it (a dbias without a dweight launch reads gm
  // with the standalone kernel, which wants the standard layout)
  const bool g_qm = dense_chain_quad_major(p, batch, in_channels, out_channels, weight) && (dbias == nullptr || dweight != nullptr) &&
                    (dweight == nullptr || (reinterpret_cast<uintptr_t>(dweight) & 31u) == 0) &&
                    ((reinterpret_cast<uintptr_t>(gy) | (p->grid16 ? 0 : reinterpret_cast<uintptr_t>(dx))) & 15u) == 0;
  SC_REQUIRE(!x_qm || p->fast != nullptr, "sc_backward_dense: quad-major saved modes without the tensor-core path");
  // the two backward contractions read the saved modes and the weight: the gy analysis pulls both into L2
  L2Prefetch pf;
  if (dweight != nullptr) { pf.ptr[0] = xm_saved; pf.bytes[0] = (unsigned long long)batch * in_channels * p->n_modes_total * sizeof(float2); }
  if (dx != nullptr) { pf.ptr[1] = weight; pf.bytes[1] = (unsigned long long)in_channels * out_channels * p->weight_elems_per_io * sizeof(float2); }
  SC_TRY(analyze(p, gy, (int64_t)batch * out_channels, gm, true, w, st, g_qm, &pf));
  SC_TRY(contract_bwd(p, reinterpret_cast<const float2*>(xm_saved), gm, reinterpret_cast<const float2*>(weight), dxm,
                      reinterpret_cast<float2*>(dweight), dbias, batch, in_channels, out_channels, st, true, x_qm, g_qm,
                      static_cast<cudaEvent_t>(grads_ready)));
  if (dx != nullptr) {
    // with a collective running on the caller's side stream (grads_ready given), the dx synthesis leaves SMs free for it
    fast_set_reserve(grads_ready != nullptr);
    const bool ok = synthesize(p, dxm, (int64_t)batch * in_channels, 0, nullptr, dx, true, w, st, g_qm);
    fast_set_reserve(false);
    SC_TRY(ok);
  }
  return 0;
}

// ---- Tucker-factorized forward / backward as ONE call each (reference _contract_tucker, :76-103) --------------------------
namespace {
struct TuckerDims {
  int d = 0, B = 0, Ci = 0, Co = 0, rf = 0, rg = 0;
  int r[SC_MAX_DIMS] = {0}, k[SC_MAX_DIMS] = {0};
  int64_t M = 1;
  // A_j: the core with axes j .. d-1 expanded to kept modes: [rf*rg][r_0..r_{j-1}][k_j..k_{d-1}]; A_d = core, A_0 = expanded weight
  int64_t chain_elems(int j) const {
    int64_t e = (int64_t)rf * rg;
    for (int l = 0; l < j; ++l) e *= r[l];
    for (int l = j; l < d; ++l) e *= k[l];
    return e;
  }
  int64_t outer(int j) const { int64_t e = (int64_t)rf * rg; for (int l = 0; l < j; ++l) e *= r[l]; return e; }
  int64_t inner(int j) const { int64_t e = 1; for (int l = j + 1; l < d; ++l) e *= k[l]; return e; }
  // saved-buffer offsets (complex elements)
  int64_t off_xm() const { return 0; }
  int64_t off_t1() const { return (int64_t)B * Ci * M; }
  int64_t off_t2() const { return off_t1() + (int64_t)B * rf * M; }
  int64_t off_wc() const { return off_t2() + (int64_t)B * rg * M; }
  int64_t off_chain(int j) const {   // A_j for 1 <= j <= d-1
    int64_t o = off_wc() + (int64_t)rf * rg * M;
    for (int l = 1; l < j; ++l) o += chain_elems(l);
    return o;
  }
  int64_t saved_elems() const { return off_chain(d); }
};

bool tucker_dims(const Plan* p, int B, int Ci, int Co, const int32_t* ranks, TuckerDims* t) {
  if (p == nullptr || ranks == nullptr || B < 1 || Ci < 1 || Co < 1) { set_error("tucker: bad arguments"); return false; }
  t->d = p->d; t->B = B; t->Ci = Ci; t->Co = Co; t->rf = ranks[0]; t->rg = ranks[1];
  t->M = p->n_modes_total;
  if (t->rf < 1 || t->rg < 1) { set_error("tucker: ranks must be >= 1"); return false; }
  for (int j = 0; j < p->d; ++j) {
    t->r[j] = ranks[2 + j]; t->k[j] = p->dim[j].k;
    if (t->r[j] < 1) { set_error("tucker: ranks must be >= 1"); return false; }
  }
  return true;
}

inline size_t a256(size_t b) { return (b + 255) & ~(size_t)255; }

struct TuckerBwdArena { float2 *g2, *g1, *dwc, *da[2]; size_t bytes; };

TuckerBwdArena tucker_bwd_arena(const TuckerDims& t, char* base) {
  TuckerBwdArena a{};
  size_t off = 0;
  auto take = [&](size_t elems) { float2* ptr = reinterpret_cast<float2*>(base + off); off += a256(elems * sizeof(float2)); return ptr; };
  a.g2 = take((size_t)t.B * t.rg * t.M);
  a.g1 = take((size_t)t.B * t.rf * t.M);
  a.dwc = take((size_t)t.rf * t.rg * t.M);
  int64_t mx = 0;
  for (int j = 0; j <= t.d; ++j) mx = std::max(mx, t.chain_elems(j));
  a.da[0] = take((size_t)mx);
  a.da[1] = take((size_t)mx);
  a.bytes = off;
  return a;
}
}  // namespace

size_t sc_tucker_saved_elems(const sc_plan* plan, int32_t batch, int32_t in_channels, int32_t out_channels, const int32_t* ranks) {
  TuckerDims t;
  if (!tucker_dims(reinterpret_cast<const Plan*>(plan), batch, in_channels, out_channels, ranks, &t)) return 0;
  return (size_t)t.saved_elems();
}

size_t sc_tucker_workspace_bytes(const sc_plan* plan, int32_t batch, int32_t in_channels, int32_t out_channels, const int32_t* ranks) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  TuckerDims t;
  if (!tucker_dims(p, batch, in_channels, out_channels, ranks, &t)) return 0;
  const int64_t n_max = (int64_t)batch * std::max(in_channels, out_channels);
  return a256(sc_workspace_bytes(plan, n_max)) + tucker_bwd_arena(t, nullptr).bytes;
}

int sc_forward_tucker(const sc_plan* plan, const sc_plan* plan_kept, const float* x, const sc_complex* core, const sc_complex* u_in,
                      const sc_complex* u_out, const sc_complex* const* u_modes, const float* bias, float* y, sc_complex* saved,
                      int32_t batch, int32_t in_channels, int32_t out_channels, const int32_t* ranks, void* workspace,
                      size_t workspace_bytes, sc_stream stream) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  const Plan* pk = reinterpret_cast<const Plan*>(plan_kept);
  SC_REQUIRE(p != nullptr && pk != nullptr && x != nullptr && core != nullptr && u_in != nullptr && u_out != nullptr && u_modes != nullptr &&
             y != nullptr && saved != nullptr, "sc_forward_tucker: null argument");
  SC_REQUIRE(pk->n_modes_total == p->n_modes_total && pk->weight_elems_per_io == p->n_modes_total,
             "sc_forward_tucker: plan_kept must be the same problem with weight extents == kept modes");
  TuckerDims t;
  SC_TRY(tucker_dims(p, batch, in_channels, out_channels, ranks, &t));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t n_max = (int64_t)t.B * std::max(t.Ci, t.Co);
  Workspace w{};
  SC_TRY(carve(p, n_max, workspace, workspace_bytes, &w));
  float2* sv = reinterpret_cast<float2*>(saved);
  float2 *xm = sv + t.off_xm(), *t1 = sv + t.off_t1(), *t2 = sv + t.off_t2(), *wc = sv + t.off_wc();
  float2* ym = w.modes[0];
  SC_TRY(analyze(p, x, (int64_t)t.B * t.Ci, xm, false, w, st));
  // expand the core along the mode axes, last axis first: A_d = core, A_j = U_j x_j A_{j+1}   (A_0 = wc)
  const float2* cur = reinterpret_cast<const float2*>(core);
  for (int j = t.d - 1; j >= 0; --j) {
    float2* dst = j == 0 ? wc : sv + t.off_chain(j);
    SC_TRY(launch_complex_table_gemm_strided(reinterpret_cast<const float2*>(u_modes[j]), t.r[j], 1, false, cur, dst, t.outer(j), t.k[j], t.r[j],
                                             (int)t.inner(j), st));
    cur = dst;
  }
  // channel mixing with U_in, the dense mode product on rank channels, channel mixing with U_out
  SC_TRY(launch_complex_table_gemm_strided(reinterpret_cast<const float2*>(u_in), 1, t.rf, false, xm, t1, t.B, t.rf, t.Ci, (int)t.M, st));
  SC_TRY(contract_fwd(pk, t1, wc, t2, t.B, t.rf, t.rg, st, false));
  SC_TRY(launch_complex_table_gemm_strided(reinterpret_cast<const float2*>(u_out), t.rg, 1, false, t2, ym, t.B, t.Co, t.rg, (int)t.M, st));
  SC_TRY(synthesize(p, ym, (int64_t)t.B * t.Co, t.Co, bias, y, false, w, st));
  return 0;
}

int sc_backward_tucker(const sc_plan* plan, const sc_plan* plan_kept, const float* gy, const sc_complex* core, const sc_complex* u_in,
                       const sc_complex* u_out, const sc_complex* const* u_modes, const sc_complex* saved, float* dx, sc_complex* d_core,
                       sc_complex* d_u_in, sc_complex* d_u_out, sc_complex* const* d_u_modes, float* dbias, int32_t batch,
                       int32_t in_channels, int32_t out_channels, const int32_t* ranks, void* workspace, size_t workspace_bytes,
                       sc_stream stream) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  const Plan* pk = reinterpret_cast<const Plan*>(plan_kept);
  SC_REQUIRE(p != nullptr && pk != nullptr && gy != nullptr && core != nullptr && u_in != nullptr && u_out != nullptr && u_modes != nullptr &&
             saved != nullptr && dx != nullptr && d_core != nullptr && d_u_in != nullptr && d_u_out != nullptr && d_u_modes != nullptr,
             "sc_backward_tucker: null argument");
  TuckerDims t;
  SC_TRY(tucker_dims(p, batch, in_channels, out_channels, ranks, &t));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t n_max = (int64_t)t.B * std::max(t.Ci, t.Co);
  const size_t tw = a256(sc_workspace_bytes(plan, n_max));
  SC_REQUIRE(workspace != nullptr && workspace_bytes >= tw + tucker_bwd_arena(t, nullptr).bytes, "sc_backward_tucker: workspace too small (see sc_tucker_workspace_bytes)");
  Workspace w{};
  SC_TRY(carve(p, n_max, workspace, tw, &w));
  TuckerBwdArena a = tucker_bwd_arena(t, static_cast<char*>(workspace) + tw);
  const float2* sv = reinterpret_cast<const float2*>(saved);
  const float2 *xm = sv + t.off_xm(), *t1 = sv + t.off_t1(), *t2 = sv + t.off_t2(), *wc = sv + t.off_wc();
  float2* gm = w.modes[0];
  float2* dxm = w.modes[1];
  SC_TRY(analyze(p, gy, (int64_t)t.B * t.Co, gm, true, w, st));
  if (dbias != nullptr) SC_TRY(launch_bias_grad(gm, dbias, t.B, t.Co, t.M, p->dc_slot, (float)(1.0 / p->s_inv), st));
  // out side: g2 = U_out^H gm,  dU_out[o, g] = sum conj(t2[b, g, m]) gm[b, o, m]
  SC_TRY(launch_complex_table_gemm_strided(reinterpret_cast<const float2*>(u_out), 1, t.rg, true, gm, a.g2, t.B, t.rg, t.Co, (int)t.M, st));
  SC_TRY(launch_pair_reduce(t2, gm, reinterpret_cast<float2*>(d_u_out), 1, t.rg, t.B, t.rg, t.Co, (int)t.M, st));
  // core side: the two mode GEMMs of the dense backward, on rank channels
  SC_TRY(contract_bwd(pk, t1, a.g2, wc, a.g1, a.dwc, nullptr, t.B, t.rf, t.rg, st, false));
  // in side
  SC_TRY(launch_pair_reduce(xm, a.g1, reinterpret_cast<float2*>(d_u_in), t.rf, 1, t.B, t.Ci, t.rf, (int)t.M, st));
  SC_TRY(launch_complex_table_gemm_strided(reinterpret_cast<const float2*>(u_in), t.rf, 1, true, a.g1, dxm, t.B, t.Ci, t.rf, (int)t.M, st));
  SC_TRY(synthesize(p, dxm, (int64_t)t.B * t.Ci, 0, nullptr, dx, true, w, st));
  // mode factors and core: undo the expansion chain, first axis first
  const float2* d_a = a.dwc;
  for (int j = 0; j < t.d; ++j) {
    const float2* a_next = (j + 1 == t.d) ? reinterpret_cast<const float2*>(core) : sv + t.off_chain(j + 1);     // A_{j+1}
    SC_TRY(launch_pair_reduce(a_next, d_a, reinterpret_cast<float2*>(d_u_modes[j]), 1, t.r[j], t.outer(j), t.r[j], t.k[j], (int)t.inner(j), st));
    float2* dst = (j + 1 == t.d) ? reinterpret_cast<float2*>(d_core) : a.da[j & 1];
    SC_TRY(launch_complex_table_gemm_strided(reinterpret_cast<const float2*>(u_modes[j]), 1, t.r[j], true, d_a, dst, t.outer(j), t.r[j], t.k[j],
                                             (int)t.inner(j), st));
    d_a = dst;
  }
  return 0;
}

int sc_allreduce_p2p(float* const* peer_buffers, uint32_t* const* peer_signal_pads, int32_t rank, int32_t world_size, int64_t n_floats,
                     float scale, int32_t n_ctas, sc_stream stream) {
  SC_REQUIRE(peer_buffers != nullptr && peer_signal_pads != nullptr, "sc_allreduce_p2p: null argument");
  SC_TRY(launch_allreduce_p2p(peer_buffers, peer_signal_pads, rank, world_size, n_floats, scale, n_ctas, static_cast<cudaStream_t>(stream)));
  return 0;
}

int sc_event_create(sc_event* event_out) {
  SC_REQUIRE(event_out != nullptr, "sc_event_create: null argument");
  cudaEvent_t ev = nullptr;
  SC_TRY(cuda_ok(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming), "cudaEventCreateWithFlags"));
  *event_out = ev;
  return 0;
}

void sc_event_destroy(sc_event event) {
  if (event != nullptr) cudaEventDestroy(static_cast<cudaEvent_t>(event));
}

int sc_stream_wait_event(sc_stream stream, sc_event event) {
  SC_REQUIRE(event != nullptr, "sc_stream_wait_event: null event");
  SC_TRY(cuda_ok(cudaStreamWaitEvent(static_cast<cudaStream_t>(stream), static_cast<cudaEvent_t>(event), 0), "cudaStreamWaitEvent"));
  return 0;
}

int sc_table_contract(const sc_complex* table, int64_t table_stride_p, int64_t table_stride_q, int conj_table,
                      const sc_complex* in, sc_complex* out, int64_t n_outer, int32_t P, int32_t Q, int32_t n_inner,
                      sc_stream stream) {
  SC_REQUIRE(table != nullptr && in != nullptr && out != nullptr, "sc_table_contract: null argument");
  SC_TRY(launch_complex_table_gemm_strided(reinterpret_cast<const float2*>(table), table_stride_p, table_stride_q, conj_table != 0,
                                           reinterpret_cast<const float2*>(in), reinterpret_cast<float2*>(out), n_outer, P, Q,
                                           n_inner, static_cast<cudaStream_t>(stream)));
  return 0;
}

int sc_pair_reduce(const sc_complex* a, const sc_complex* b, sc_complex* out, int64_t out_stride_p, int64_t out_stride_q,
                   int64_t n_outer, int32_t P, int32_t Q, int32_t n_inner, sc_stream stream) {
  SC_REQUIRE(a != nullptr && b != nullptr && out != nullptr, "sc_pair_reduce: null argument");
  SC_TRY(launch_pair_reduce(reinterpret_cast<const float2*>(a), reinterpret_cast<const float2*>(b), reinterpret_cast<float2*>(out),
                            out_stride_p, out_stride_q, n_outer, P, Q, n_inner, static_cast<cudaStream_t>(stream)));
  return 0;
}

static bool cp_args(const sc_complex* const* factors, const int32_t* kept, int32_t ndim, const float2** u, int* k) {
  if (factors == nullptr || kept == nullptr || ndim < 1 || ndim > SC_MAX_DIMS) { set_error("cp: bad factor arguments"); return false; }
  for (int j = 0; j < ndim; ++j) { u[j] = reinterpret_cast<const float2*>(factors[j]); k[j] = kept[j]; }
  return true;
}

int sc_cp_scale(const sc_complex* const* mode_factors, const int32_t* kept, int32_t ndim, const sc_complex* lambda,
                sc_complex* scale, int32_t rank, sc_stream stream) {
  const float2* u[SC_MAX_DIMS]; int k[SC_MAX_DIMS];
  SC_TRY(cp_args(mode_factors, kept, ndim, u, k));
  int64_t M = 1; for (int j = 0; j < ndim; ++j) M *= k[j];
  SC_TRY(launch_cp_scale(u, k, ndim, reinterpret_cast<const float2*>(lambda), reinterpret_cast<float2*>(scale), rank, M,
                         static_cast<cudaStream_t>(stream)));
  return 0;
}

int sc_cp_apply(const sc_complex* in, const sc_complex* scale, sc_complex* out, int conj_scale, int32_t batch,
                int64_t per_batch, sc_stream stream) {
  SC_REQUIRE(in != nullptr && scale != nullptr && out != nullptr, "sc_cp_apply: null argument");
  SC_TRY(launch_cp_apply(reinterpret_cast<const float2*>(in), reinterpret_cast<const float2*>(scale), reinterpret_cast<float2*>(out),
                         conj_scale != 0, batch, per_batch, static_cast<cudaStream_t>(stream)));
  return 0;
}

int sc_cp_dscale(const sc_complex* t, const sc_complex* g, sc_complex* dscale, int32_t batch, int64_t per_batch,
                 sc_stream stream) {
  SC_REQUIRE(t != nullptr && g != nullptr && dscale != nullptr, "sc_cp_dscale: null argument");
  SC_TRY(launch_cp_dscale(reinterpret_cast<const float2*>(t), reinterpret_cast<const float2*>(g), reinterpret_cast<float2*>(dscale),
                          batch, per_batch, static_cast<cudaStream_t>(stream)));
  return 0;
}

int sc_cp_factor_grad(const sc_complex* const* mode_factors, const int32_t* kept, int32_t ndim, const sc_complex* lambda,
                      const sc_complex* dscale, sc_complex* out, int32_t which, int32_t rank, sc_stream stream) {
  const float2* u[SC_MAX_DIMS]; int k[SC_MAX_DIMS];
  SC_TRY(cp_args(mode_factors, kept, ndim, u, k));
  SC_REQUIRE(which >= -1 && which < ndim, "sc_cp_factor_grad: bad factor index");
  int64_t M = 1; for (int j = 0; j < ndim; ++j) M *= k[j];
  SC_TRY(launch_cp_factor_grad(u, k, ndim, reinterpret_cast<const float2*>(lambda), reinterpret_cast<const float2*>(dscale),
                               reinterpret_cast<float2*>(out), which, rank, M, static_cast<cudaStream_t>(stream)));
  return 0;
}

// ---- dry run of the CP / TT chains (test hook) ------------------------------------------------------------------------------
// The chain entry points below are sequences of primitive launches whose only own logic is WHICH buffer (offset into the saved
// buffer / workspace / a parameter) goes WHERE with WHICH strides.  With a recorder installed (sc_hostcheck_chain_log) every
// primitive call of a chain is appended to a log -- opcode, argument count, arguments (pointers as integers) -- instead of being
// launched, so that the CPU test tier can replay the log on host arrays and compare the result with the oracle: the orchestration
// is checked without a GPU, the primitives themselves are validated on hardware.
extern "C++" {
namespace {
enum { CH_ANALYZE = 1, CH_SYNTHESIZE, CH_TABLE, CH_PAIR, CH_CP_SCALE, CH_CP_APPLY, CH_CP_DSCALE, CH_CP_FACTOR_GRAD, CH_BIAS_GRAD,
       CH_CONTRACT_FWD, CH_CONTRACT_BWD };
thread_local std::vector<int64_t>* t_chain_log = nullptr;

inline int64_t ch_word(const void* ptr) { return (int64_t)reinterpret_cast<uintptr_t>(ptr); }
inline int64_t ch_word(int64_t v) { return v; }
inline int64_t ch_word(int v) { return v; }
inline int64_t ch_word(bool v) { return v ? 1 : 0; }
inline int64_t ch_word(float v) { int64_t w = 0; std::memcpy(&w, &v, sizeof(float)); return w; }
template <class... A>
void ch_log(int op, A... a) {
  t_chain_log->push_back(op);
  t_chain_log->push_back((int64_t)sizeof...(A));
  (t_chain_log->push_back(ch_word(a)), ...);
}

bool ch_analyze(const Plan* p, const float* images, int64_t n_images, float2* modes_out, bool adjoint, const Workspace& w,
                cudaStream_t st) {
  if (t_chain_log != nullptr) { ch_log(CH_ANALYZE, images, n_images, modes_out, adjoint); return true; }
  return analyze(p, images, n_images, modes_out, adjoint, w, st);
}
bool ch_synthesize(const Plan* p, const float2* modes_in, int64_t n_images, int n_channels, const float* bias, float* images_out,
                   bool adjoint, const Workspace& w, cudaStream_t st) {
  if (t_chain_log != nullptr) { ch_log(CH_SYNTHESIZE, modes_in, n_images, n_channels, bias, images_out, adjoint); return true; }
  return synthesize(p, modes_in, n_images, n_channels, bias, images_out, adjoint, w, st);
}
bool ch_table(const float2* T, int64_t sTp, int64_t sTq, bool conjT, const float2* in, float2* out, int64_t O, int P, int Q, int I,
              cudaStream_t st) {
  if (t_chain_log != nullptr) { ch_log(CH_TABLE, T, sTp, sTq, conjT, in, out, O, P, Q, I); return true; }
  return launch_complex_table_gemm_strided(T, sTp, sTq, conjT, in, out, O, P, Q, I, st);
}
bool ch_pair(const float2* A, const float2* B, float2* out, int64_t sOp, int64_t sOq, int64_t O, int P, int Q, int I, cudaStream_t st) {
  if (t_chain_log != nullptr) { ch_log(CH_PAIR, A, B, out, sOp, sOq, O, P, Q, I); return true; }
  return launch_pair_reduce(A, B, out, sOp, sOq, O, P, Q, I, st);
}
bool ch_cp_scale(const float2* const* u, const int* k, int d, const float2* lambda, float2* scale, int R, int64_t M, cudaStream_t st) {
  if (t_chain_log != nullptr) {
    ch_log(CH_CP_SCALE, d, u[0], d > 1 ? u[1] : nullptr, d > 2 ? u[2] : nullptr, d > 3 ? u[3] : nullptr, k[0], d > 1 ? k[1] : 0,
           d > 2 ? k[2] : 0, d > 3 ? k[3] : 0, lambda, scale, R, M);
    return true;
  }
  return launch_cp_scale(u, k, d, lambda, scale, R, M, st);
}
bool ch_cp_apply(const float2* in, const float2* scale, float2* out, bool conj_scale, int batch, int64_t per_batch, cudaStream_t st) {
  if (t_chain_log != nullptr) { ch_log(CH_CP_APPLY, in, scale, out, conj_scale, batch, per_batch); return true; }
  return launch_cp_apply(in, scale, out, conj_scale, batch, per_batch, st);
}
bool ch_cp_dscale(const float2* t, const float2* g, float2* dscale, int batch, int64_t per_batch, cudaStream_t st) {
  if (t_chain_log != nullptr) { ch_log(CH_CP_DSCALE, t, g, dscale, batch, per_batch); return true; }
  return launch_cp_dscale(t, g, dscale, batch, per_batch, st);
}
bool ch_cp_factor_grad(const float2* const* u, const int* k, int d, const float2* lambda, const float2* dscale, float2* out, int which,
                       int R, int64_t M, cudaStream_t st) {
  if (t_chain_log != nullptr) {
    ch_log(CH_CP_FACTOR_GRAD, d, u[0], d > 1 ? u[1] : nullptr, d > 2 ? u[2] : nullptr, d > 3 ? u[3] : nullptr, k[0], d > 1 ? k[1] : 0,
           d > 2 ? k[2] : 0, d > 3 ? k[3] : 0, lambda, dscale, out, which, R, M);
    return true;
  }
  return launch_cp_factor_grad(u, k, d, lambda, dscale, out, which, R, M, st);
}
bool ch_bias_grad(const float2* gm, float* dbias, int batch, int out_channels, int64_t n_modes, int dc_slot, float inv_scale,
                  cudaStream_t st) {
  if (t_chain_log != nullptr) { ch_log(CH_BIAS_GRAD, gm, dbias, batch, out_channels, n_modes, dc_slot, inv_scale); return true; }
  return launch_bias_grad(gm, dbias, batch, out_channels, n_modes, dc_slot, inv_scale, st);
}
bool ch_contract_fwd(const Plan* p, const float2* xm, const float2* w, float2* ym, int B, int Ci, int Co, cudaStream_t st) {
  if (t_chain_log != nullptr) { ch_log(CH_CONTRACT_FWD, xm, w, ym, B, Ci, Co); return true; }
  return contract_fwd(p, xm, w, ym, B, Ci, Co, st, false);
}
bool ch_contract_bwd(const Plan* p, const float2* xm, const float2* gm, const float2* w, float2* dxm, float2* dw, int B, int Ci, int Co,
                     cudaStream_t st) {
  if (t_chain_log != nullptr) { ch_log(CH_CONTRACT_BWD, xm, gm, w, dxm, dw, B, Ci, Co); return true; }
  return contract_bwd(p, xm, gm, w, dxm, dw, nullptr, B, Ci, Co, st, false);
}
}  // namespace
}  // extern "C++"

// ---- CP-factorized forward / backward as ONE call each (reference _contract_cp, :55-73) -----------------------------------
// The same launches, in the same order and with the same operands, as the Python-orchestrated chain (`_SpectralConvCP`,
// neuraloperator_b200/spectral_conv.py), issued from one saved buffer and one workspace.
namespace {
struct CpDims {
  int d = 0, B = 0, Ci = 0, Co = 0, R = 0;
  int k[SC_MAX_DIMS] = {0};
  int64_t M = 1;
  // saved-buffer offsets (complex elements): kept input modes | x U_in | (x U_in) * scale | scale
  int64_t off_t1() const { return (int64_t)B * Ci * M; }
  int64_t off_t2() const { return off_t1() + (int64_t)B * R * M; }
  int64_t off_scale() const { return off_t2() + (int64_t)B * R * M; }
  int64_t saved_elems() const { return off_scale() + (int64_t)R * M; }
};

bool cp_dims(const Plan* p, int B, int Ci, int Co, int R, CpDims* t) {
  if (p == nullptr || B < 1 || Ci < 1 || Co < 1 || R < 1) { set_error("cp: bad arguments"); return false; }
  t->d = p->d; t->B = B; t->Ci = Ci; t->Co = Co; t->R = R; t->M = p->n_modes_total;
  for (int j = 0; j < p->d; ++j) t->k[j] = p->dim[j].k;
  return true;
}

struct CpBwdArena { float2 *g2, *g1, *dscale; size_t bytes; };

CpBwdArena cp_bwd_arena(const CpDims& t, char* base) {
  CpBwdArena a{};
  size_t off = 0;
  auto take = [&](size_t elems) { float2* ptr = reinterpret_cast<float2*>(base + off); off += a256(elems * sizeof(float2)); return ptr; };
  a.g2 = take((size_t)t.B * t.R * t.M);
  a.g1 = take((size_t)t.B * t.R * t.M);
  a.dscale = take((size_t)t.R * t.M);
  a.bytes = off;
  return a;
}
}  // namespace

size_t sc_cp_saved_elems(const sc_plan* plan, int32_t batch, int32_t in_channels, int32_t out_channels, int32_t rank) {
  CpDims t;
  if (!cp_dims(reinterpret_cast<const Plan*>(plan), batch, in_channels, out_channels, rank, &t)) return 0;
  return (size_t)t.saved_elems();
}

size_t sc_cp_workspace_bytes(const sc_plan* plan, int32_t batch, int32_t in_channels, int32_t out_channels, int32_t rank) {
  CpDims t;
  if (!cp_dims(reinterpret_cast<const Plan*>(plan), batch, in_channels, out_channels, rank, &t)) return 0;
  const int64_t n_max = (int64_t)batch * std::max(in_channels, out_channels);
  return a256(sc_workspace_bytes(plan, n_max)) + cp_bwd_arena(t, nullptr).bytes;
}

int sc_forward_cp(const sc_plan* plan, const float* x, const sc_complex* lambda, const sc_complex* u_in, const sc_complex* u_out,
                  const sc_complex* const* u_modes, const float* bias, float* y, sc_complex* saved, int32_t batch, int32_t in_channels,
                  int32_t out_channels, int32_t rank, void* workspace, size_t workspace_bytes, sc_stream stream) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  SC_REQUIRE(p != nullptr && x != nullptr && lambda != nullptr && u_in != nullptr && u_out != nullptr && u_modes != nullptr && y != nullptr &&
             saved != nullptr, "sc_forward_cp: null argument");
  CpDims t;
  SC_TRY(cp_dims(p, batch, in_channels, out_channels, rank, &t));
  const float2* u[SC_MAX_DIMS]; int k[SC_MAX_DIMS];
  SC_TRY(cp_args(u_modes, t.k, t.d, u, k));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t n_max = (int64_t)t.B * std::max(t.Ci, t.Co);
  Workspace w{};
  SC_TRY(carve(p, n_max, workspace, workspace_bytes, &w));
  float2* sv = reinterpret_cast<float2*>(saved);
  float2 *xm = sv, *t1 = sv + t.off_t1(), *t2 = sv + t.off_t2(), *scale = sv + t.off_scale();
  float2* ym = w.modes[0];
  SC_TRY(ch_analyze(p, x, (int64_t)t.B * t.Ci, xm, false, w, st));
  SC_TRY(ch_cp_scale(u, k, t.d, reinterpret_cast<const float2*>(lambda), scale, t.R, t.M, st));
  // T[p = e, q = i] = U_in[i, e];  pointwise scale;  T[p = o, q = e] = U_out[o, e]
  SC_TRY(ch_table(reinterpret_cast<const float2*>(u_in), 1, t.R, false, xm, t1, t.B, t.R, t.Ci, (int)t.M, st));
  SC_TRY(ch_cp_apply(t1, scale, t2, false, t.B, (int64_t)t.R * t.M, st));
  SC_TRY(ch_table(reinterpret_cast<const float2*>(u_out), t.R, 1, false, t2, ym, t.B, t.Co, t.R, (int)t.M, st));
  SC_TRY(ch_synthesize(p, ym, (int64_t)t.B * t.Co, t.Co, bias, y, false, w, st));
  return 0;
}

int sc_backward_cp(const sc_plan* plan, const float* gy, const sc_complex* lambda, const sc_complex* u_in, const sc_complex* u_out,
                   const sc_complex* const* u_modes, const sc_complex* saved, float* dx, sc_complex* d_lambda, sc_complex* d_u_in,
                   sc_complex* d_u_out, sc_complex* const* d_u_modes, float* dbias, int32_t batch, int32_t in_channels,
                   int32_t out_channels, int32_t rank, void* workspace, size_t workspace_bytes, sc_stream stream) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  SC_REQUIRE(p != nullptr && gy != nullptr && lambda != nullptr && u_in != nullptr && u_out != nullptr && u_modes != nullptr &&
             saved != nullptr && dx != nullptr && d_lambda != nullptr && d_u_in != nullptr && d_u_out != nullptr && d_u_modes != nullptr,
             "sc_backward_cp: null argument");
  CpDims t;
  SC_TRY(cp_dims(p, batch, in_channels, out_channels, rank, &t));
  const float2* u[SC_MAX_DIMS]; int k[SC_MAX_DIMS];
  SC_TRY(cp_args(u_modes, t.k, t.d, u, k));
  for (int j = 0; j < t.d; ++j) SC_REQUIRE(d_u_modes[j] != nullptr, "sc_backward_cp: null mode-factor gradient");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t n_max = (int64_t)t.B * std::max(t.Ci, t.Co);
  const size_t tw = a256(sc_workspace_bytes(plan, n_max));
  SC_REQUIRE(workspace != nullptr && workspace_bytes >= tw + cp_bwd_arena(t, nullptr).bytes, "sc_backward_cp: workspace too small (see sc_cp_workspace_bytes)");
  Workspace w{};
  SC_TRY(carve(p, n_max, workspace, tw, &w));
  CpBwdArena a = cp_bwd_arena(t, static_cast<char*>(workspace) + tw);
  const float2* sv = reinterpret_cast<const float2*>(saved);
  const float2 *xm = sv, *t1 = sv + t.off_t1(), *t2 = sv + t.off_t2(), *scale = sv + t.off_scale();
  const float2* lam = reinterpret_cast<const float2*>(lambda);
  float2* gm = w.modes[0];
  float2* dxm = w.modes[1];
  const int64_t per = (int64_t)t.R * t.M;
  SC_TRY(ch_analyze(p, gy, (int64_t)t.B * t.Co, gm, true, w, st));
  if (dbias != nullptr) SC_TRY(ch_bias_grad(gm, dbias, t.B, t.Co, t.M, p->dc_slot, (float)(1.0 / p->s_inv), st));
  // out side: g2 = U_out^H gm,  dU_out[o, e] = sum conj(t2[b, e, m]) gm[b, o, m]
  SC_TRY(ch_table(reinterpret_cast<const float2*>(u_out), 1, t.R, true, gm, a.g2, t.B, t.R, t.Co, (int)t.M, st));
  SC_TRY(ch_pair(t2, gm, reinterpret_cast<float2*>(d_u_out), 1, t.R, t.B, t.R, t.Co, (int)t.M, st));
  // pointwise stage: dscale = sum_b conj(t1) g2,  g1 = g2 conj(scale)
  SC_TRY(ch_cp_dscale(t1, a.g2, a.dscale, t.B, per, st));
  SC_TRY(ch_cp_apply(a.g2, scale, a.g1, true, t.B, per, st));
  // in side
  SC_TRY(ch_pair(xm, a.g1, reinterpret_cast<float2*>(d_u_in), t.R, 1, t.B, t.Ci, t.R, (int)t.M, st));
  SC_TRY(ch_table(reinterpret_cast<const float2*>(u_in), t.R, 1, true, a.g1, dxm, t.B, t.Ci, t.R, (int)t.M, st));
  SC_TRY(ch_synthesize(p, dxm, (int64_t)t.B * t.Ci, 0, nullptr, dx, true, w, st));
  // lambda and the mode factors from dscale
  SC_TRY(ch_cp_factor_grad(u, k, t.d, lam, a.dscale, reinterpret_cast<float2*>(d_lambda), -1, t.R, t.M, st));
  for (int j = 0; j < t.d; ++j)
    SC_TRY(ch_cp_factor_grad(u, k, t.d, lam, a.dscale, reinterpret_cast<float2*>(d_u_modes[j]), j, t.R, t.M, st));
  return 0;
}

// ---- TT-factorized forward / backward as ONE call each (reference _contract_tt, :106-127) ---------------------------------
// W[i,o,m] = G0[0,i,:] G1[:,o,:] C_0[:,m_0,:] .. C_{d-1}[:,m_{d-1},0].  ranks = {r1, r_0 .. r_{d-1}}: G0 (1, Ci, r1), G1 (r1, Co, r_0),
// cores[j] = the KEPT rows of mode core j, contiguous (r_j, k_j, r_{j+1}) with r_d = 1.  Same launches, order and operands as the
// Python-orchestrated chain (`_SpectralConvTT`): the mode cores are multiplied right to left into V[r_0, m]; G1 V is a rank-r1 weight
// block that the dense mode GEMM applies to xm G0.
namespace {
struct TtDims {
  int d = 0, B = 0, Ci = 0, Co = 0, r1 = 0;
  int r[SC_MAX_DIMS + 1] = {0}, k[SC_MAX_DIMS] = {0};      // r[j]: left rank of mode core j, r[d] = 1
  int64_t M = 1;
  int64_t inner(int j) const { int64_t e = 1; for (int l = j + 1; l < d; ++l) e *= k[l]; return e; }      // prod_{l > j} k_l
  int64_t chain_elems(int j) const { return (int64_t)r[j] * k[j] * inner(j); }                            // A_j: (r_j, k_j .. k_{d-1})
  // saved-buffer offsets (complex elements): kept input modes | xm G0 | G1 V | A_{d-2}, .., A_0 (A_{d-1} is cores[d-1] itself)
  int64_t off_t1() const { return (int64_t)B * Ci * M; }
  int64_t off_wc() const { return off_t1() + (int64_t)B * r1 * M; }
  int64_t off_chain(int j) const {       // 0 <= j <= d-2
    int64_t o = off_wc() + (int64_t)r1 * Co * M;
    for (int l = d - 2; l > j; --l) o += chain_elems(l);
    return o;
  }
  int64_t saved_elems() const { return d >= 2 ? off_chain(0) + chain_elems(0) : off_wc() + (int64_t)r1 * Co * M; }
};

bool tt_dims(const Plan* p, int B, int Ci, int Co, const int32_t* ranks, TtDims* t) {
  if (p == nullptr || ranks == nullptr || B < 1 || Ci < 1 || Co < 1) { set_error("tt: bad arguments"); return false; }
  t->d = p->d; t->B = B; t->Ci = Ci; t->Co = Co; t->r1 = ranks[0]; t->M = p->n_modes_total;
  if (t->r1 < 1) { set_error("tt: ranks must be >= 1"); return false; }
  for (int j = 0; j < p->d; ++j) {
    t->r[j] = ranks[1 + j]; t->k[j] = p->dim[j].k;
    if (t->r[j] < 1) { set_error("tt: ranks must be >= 1"); return false; }
  }
  t->r[p->d] = 1;
  return true;
}

struct TtBwdArena { float2 *g1, *dwc, *da[2]; size_t bytes; };

TtBwdArena tt_bwd_arena(const TtDims& t, char* base) {
  TtBwdArena a{};
  size_t off = 0;
  auto take = [&](size_t elems) { float2* ptr = reinterpret_cast<float2*>(base + off); off += a256(elems * sizeof(float2)); return ptr; };
  a.g1 = take((size_t)t.B * t.r1 * t.M);
  a.dwc = take((size_t)t.r1 * t.Co * t.M);
  int64_t mx = 0;
  for (int j = 0; j < t.d; ++j) mx = std::max(mx, t.chain_elems(j));
  a.da[0] = take((size_t)mx);
  a.da[1] = take((size_t)mx);
  a.bytes = off;
  return a;
}
}  // namespace

size_t sc_tt_saved_elems(const sc_plan* plan, int32_t batch, int32_t in_channels, int32_t out_channels, const int32_t* ranks) {
  TtDims t;
  if (!tt_dims(reinterpret_cast<const Plan*>(plan), batch, in_channels, out_channels, ranks, &t)) return 0;
  return (size_t)t.saved_elems();
}

size_t sc_tt_workspace_bytes(const sc_plan* plan, int32_t batch, int32_t in_channels, int32_t out_channels, const int32_t* ranks) {
  TtDims t;
  if (!tt_dims(reinterpret_cast<const Plan*>(plan), batch, in_channels, out_channels, ranks, &t)) return 0;
  const int64_t n_max = (int64_t)batch * std::max(in_channels, out_channels);
  return a256(sc_workspace_bytes(plan, n_max)) + tt_bwd_arena(t, nullptr).bytes;
}

int sc_forward_tt(const sc_plan* plan, const sc_plan* plan_kept, const float* x, const sc_complex* g0, const sc_complex* g1,
                  const sc_complex* const* cores, const float* bias, float* y, sc_complex* saved, int32_t batch, int32_t in_channels,
                  int32_t out_channels, const int32_t* ranks, void* workspace, size_t workspace_bytes, sc_stream stream) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  const Plan* pk = reinterpret_cast<const Plan*>(plan_kept);
  SC_REQUIRE(p != nullptr && pk != nullptr && x != nullptr && g0 != nullptr && g1 != nullptr && cores != nullptr && y != nullptr &&
             saved != nullptr, "sc_forward_tt: null argument");
  SC_REQUIRE(pk->n_modes_total == p->n_modes_total && pk->weight_elems_per_io == p->n_modes_total,
             "sc_forward_tt: plan_kept must be the same problem with weight extents == kept modes");
  TtDims t;
  SC_TRY(tt_dims(p, batch, in_channels, out_channels, ranks, &t));
  for (int j = 0; j < t.d; ++j) SC_REQUIRE(cores[j] != nullptr, "sc_forward_tt: null mode core");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t n_max = (int64_t)t.B * std::max(t.Ci, t.Co);
  Workspace w{};
  SC_TRY(carve(p, n_max, workspace, workspace_bytes, &w));
  float2* sv = reinterpret_cast<float2*>(saved);
  float2 *xm = sv, *t1 = sv + t.off_t1(), *wc = sv + t.off_wc();
  float2* ym = w.modes[0];
  SC_TRY(ch_analyze(p, x, (int64_t)t.B * t.Ci, xm, false, w, st));
  // A_{d-1} = cores[d-1] (r_{d-1}, k_{d-1});  A_j[(a, m_j), rest] = sum_b C_j[a, m_j, b] A_{j+1}[b, rest];  V = A_0 (r_0, M)
  const float2* cur = reinterpret_cast<const float2*>(cores[t.d - 1]);
  for (int j = t.d - 2; j >= 0; --j) {
    float2* dst = sv + t.off_chain(j);
    SC_TRY(ch_table(reinterpret_cast<const float2*>(cores[j]), t.r[j + 1], 1, false, cur, dst, 1, t.r[j] * t.k[j],
                                             t.r[j + 1], (int)t.inner(j), st));
    cur = dst;
  }
  // wc[(r, o), m] = sum_s G1[r, o, s] V[s, m];  t1 = xm G0;  dense mode product on the r1 rank channels
  SC_TRY(ch_table(reinterpret_cast<const float2*>(g1), t.r[0], 1, false, cur, wc, 1, t.r1 * t.Co, t.r[0], (int)t.M, st));
  SC_TRY(ch_table(reinterpret_cast<const float2*>(g0), 1, t.r1, false, xm, t1, t.B, t.r1, t.Ci, (int)t.M, st));
  SC_TRY(ch_contract_fwd(pk, t1, wc, ym, t.B, t.r1, t.Co, st));
  SC_TRY(ch_synthesize(p, ym, (int64_t)t.B * t.Co, t.Co, bias, y, false, w, st));
  return 0;
}

int sc_backward_tt(const sc_plan* plan, const sc_plan* plan_kept, const float* gy, const sc_complex* g0, const sc_complex* g1,
                   const sc_complex* const* cores, const sc_complex* saved, float* dx, sc_complex* d_g0, sc_complex* d_g1,
                   sc_complex* const* d_cores, float* dbias, int32_t batch, int32_t in_channels, int32_t out_channels, const int32_t* ranks,
                   void* workspace, size_t workspace_bytes, sc_stream stream) {
  const Plan* p = reinterpret_cast<const Plan*>(plan);
  const Plan* pk = reinterpret_cast<const Plan*>(plan_kept);
  SC_REQUIRE(p != nullptr && pk != nullptr && gy != nullptr && g0 != nullptr && g1 != nullptr && cores != nullptr && saved != nullptr &&
             dx != nullptr && d_g0 != nullptr && d_g1 != nullptr && d_cores != nullptr, "sc_backward_tt: null argument");
  TtDims t;
  SC_TRY(tt_dims(p, batch, in_channels, out_channels, ranks, &t));
  for (int j = 0; j < t.d; ++j) SC_REQUIRE(cores[j] != nullptr && d_cores[j] != nullptr, "sc_backward_tt: null mode core / gradient");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t n_max = (int64_t)t.B * std::max(t.Ci, t.Co);
  const size_t tw = a256(sc_workspace_bytes(plan, n_max));
  SC_REQUIRE(workspace != nullptr && workspace_bytes >= tw + tt_bwd_arena(t, nullptr).bytes, "sc_backward_tt: workspace too small (see sc_tt_workspace_bytes)");
  Workspace w{};
  SC_TRY(carve(p, n_max, workspace, tw, &w));
  TtBwdArena a = tt_bwd_arena(t, static_cast<char*>(workspace) + tw);
  const float2* sv = reinterpret_cast<const float2*>(saved);
  const float2 *xm = sv, *t1 = sv + t.off_t1(), *wc = sv + t.off_wc();
  float2* gm = w.modes[0];
  float2* dxm = w.modes[1];
  SC_TRY(ch_analyze(p, gy, (int64_t)t.B * t.Co, gm, true, w, st));
  if (dbias != nullptr) SC_TRY(ch_bias_grad(gm, dbias, t.B, t.Co, t.M, p->dc_slot, (float)(1.0 / p->s_inv), st));
  // the two mode GEMMs of the dense backward on the rank channels: g1 = d(t1), dwc = d(wc)
  SC_TRY(ch_contract_bwd(pk, t1, gm, wc, a.g1, a.dwc, t.B, t.r1, t.Co, st));
  // in side: dG0[0, i, r] = sum conj(xm[b, i, m]) g1[b, r, m];  dxm = g1 G0^H
  SC_TRY(ch_pair(xm, a.g1, reinterpret_cast<float2*>(d_g0), t.r1, 1, t.B, t.Ci, t.r1, (int)t.M, st));
  SC_TRY(ch_table(reinterpret_cast<const float2*>(g0), t.r1, 1, true, a.g1, dxm, t.B, t.Ci, t.r1, (int)t.M, st));
  SC_TRY(ch_synthesize(p, dxm, (int64_t)t.B * t.Ci, 0, nullptr, dx, true, w, st));
  // weight side: dG1[(r, o), s] = sum_m conj(V[s, m]) dwc[(r, o), m];  dV = G1^H dwc;  then undo the chain, first axis first
  const float2* v = t.d >= 2 ? sv + t.off_chain(0) : reinterpret_cast<const float2*>(cores[0]);
  SC_TRY(ch_pair(v, a.dwc, reinterpret_cast<float2*>(d_g1), 1, t.r[0], 1, t.r[0], t.r1 * t.Co, (int)t.M, st));
  float2* d_a = t.d == 1 ? reinterpret_cast<float2*>(d_cores[0]) : a.da[0];
  SC_TRY(ch_table(reinterpret_cast<const float2*>(g1), 1, t.r[0], true, a.dwc, d_a, 1, t.r[0], t.r1 * t.Co, (int)t.M, st));
  for (int j = 0; j + 1 < t.d; ++j) {
    const float2* a_next = (j + 1 == t.d - 1) ? reinterpret_cast<const float2*>(cores[t.d - 1]) : sv + t.off_chain(j + 1);     // A_{j+1}: (r_{j+1}, inner)
    const int64_t inner = t.inner(j);
    SC_TRY(ch_pair(a_next, d_a, reinterpret_cast<float2*>(d_cores[j]), 1, t.r[j + 1], 1, t.r[j + 1], t.r[j] * t.k[j], (int)inner, st));
    float2* dst = (j + 1 == t.d - 1) ? reinterpret_cast<float2*>(d_cores[t.d - 1]) : a.da[(j + 1) & 1];
    SC_TRY(ch_table(reinterpret_cast<const float2*>(cores[j]), 1, t.r[j + 1], true, d_a, dst, 1, t.r[j + 1],
                                             t.r[j] * t.k[j], (int)inner, st));
    d_a = dst;
  }
  return 0;
}

// ---- test hook: the launch sequence of a CP / TT chain for `problem`, recorded instead of executed (no device needed) ------------
// kind 0 = CP (ranks[0] = R), 1 = TT (ranks = {r1, r_0 .. r_{d-1}}); direction 0 = forward, 1 = backward.  Buffers are given as
// synthetic addresses (region << 40): 1 x / gy, 2 y / dx, 3 saved, 4 workspace, 5 lambda, 6 u_in / g0, 7 u_out / g1, 8+j mode factor /
// core j, 12 bias / dbias, 15 d_lambda, 16 d_u_in / d_g0, 17 d_u_out / d_g1, 18+j gradient of mode factor / core j.
// log_out receives {opcode, n_args, args...} records (see the CH_* enum and the ch_* wrappers); returns the number of words.
int sc_hostcheck_chain_log(const sc_problem* problem, int kind, int direction, int32_t batch, int32_t in_channels, int32_t out_channels,
                           const int32_t* ranks, int64_t* log_out, size_t capacity_words, int64_t* n_words_out) {
  SC_REQUIRE(problem != nullptr && ranks != nullptr && n_words_out != nullptr, "sc_hostcheck_chain_log: null argument");
  SC_REQUIRE((kind == 0 || kind == 1) && (direction == 0 || direction == 1), "sc_hostcheck_chain_log: bad kind / direction");
  Plan plan, plan_kept;
  plan.host_only = true;
  plan_kept.host_only = true;
  SC_TRY(build_plan(*problem, &plan));
  sc_problem pk = *problem;
  for (int j = 0; j < plan.d; ++j) { pk.n_modes[j] = plan.dim[j].k; pk.max_n_modes[j] = plan.dim[j].k; }
  SC_TRY(build_plan(pk, &plan_kept));
  auto at = [](int region) { return reinterpret_cast<void*>((uintptr_t)region << 40); };
  const sc_complex* modes_in[SC_MAX_DIMS];
  sc_complex* modes_out[SC_MAX_DIMS];
  for (int j = 0; j < SC_MAX_DIMS; ++j) { modes_in[j] = static_cast<const sc_complex*>(at(8 + j)); modes_out[j] = static_cast<sc_complex*>(at(18 + j)); }
  const sc_plan* P = reinterpret_cast<const sc_plan*>(&plan);
  const sc_plan* PK = reinterpret_cast<const sc_plan*>(&plan_kept);
  std::vector<int64_t> log;
  // record 0: what the Python side allocates for this chain (the replay checks every access against these bounds)
  const size_t saved_elems = kind == 0 ? sc_cp_saved_elems(P, batch, in_channels, out_channels, ranks[0])
                                       : sc_tt_saved_elems(P, batch, in_channels, out_channels, ranks);
  const size_t ws_bytes = kind == 0 ? sc_cp_workspace_bytes(P, batch, in_channels, out_channels, ranks[0])
                                    : sc_tt_workspace_bytes(P, batch, in_channels, out_channels, ranks);
  log.push_back(0); log.push_back(2); log.push_back((int64_t)saved_elems); log.push_back((int64_t)ws_bytes);
  t_chain_log = &log;
  int rc = 0;
  if (kind == 0 && direction == 0)
    rc = sc_forward_cp(P, static_cast<const float*>(at(1)), static_cast<const sc_complex*>(at(5)), static_cast<const sc_complex*>(at(6)),
                       static_cast<const sc_complex*>(at(7)), modes_in, static_cast<const float*>(at(12)), static_cast<float*>(at(2)),
                       static_cast<sc_complex*>(at(3)), batch, in_channels, out_channels, ranks[0], at(4), ws_bytes, nullptr);
  else if (kind == 0)
    rc = sc_backward_cp(P, static_cast<const float*>(at(1)), static_cast<const sc_complex*>(at(5)), static_cast<const sc_complex*>(at(6)),
                        static_cast<const sc_complex*>(at(7)), modes_in, static_cast<const sc_complex*>(at(3)), static_cast<float*>(at(2)),
                        static_cast<sc_complex*>(at(15)), static_cast<sc_complex*>(at(16)), static_cast<sc_complex*>(at(17)), modes_out,
                        static_cast<float*>(at(12)), batch, in_channels, out_channels, ranks[0], at(4), ws_bytes, nullptr);
  else if (direction == 0)
    rc = sc_forward_tt(P, PK, static_cast<const float*>(at(1)), static_cast<const sc_complex*>(at(6)), static_cast<const sc_complex*>(at(7)),
                       modes_in, static_cast<const float*>(at(12)), static_cast<float*>(at(2)), static_cast<sc_complex*>(at(3)), batch,
                       in_channels, out_channels, ranks, at(4), ws_bytes, nullptr);
  else
    rc = sc_backward_tt(P, PK, static_cast<const float*>(at(1)), static_cast<const sc_complex*>(at(6)), static_cast<const sc_complex*>(at(7)),
                        modes_in, static_cast<const sc_complex*>(at(3)), static_cast<float*>(at(2)), static_cast<sc_complex*>(at(16)),
                        static_cast<sc_complex*>(at(17)), modes_out, static_cast<float*>(at(12)), batch, in_channels, out_channels, ranks,
                        at(4), ws_bytes, nullptr);
  t_chain_log = nullptr;
  if (rc != 0) return rc;
  *n_words_out = (int64_t)log.size();
  if (log_out != nullptr) {
    SC_REQUIRE(log.size() <= capacity_words, "sc_hostcheck_chain_log: log buffer too small");
    std::memcpy(log_out, log.data(), log.size() * sizeof(int64_t));
  }
  return 0;
}

int sc_selftest_umma(const float* a, const float* b, float* d, int32_t n, int32_t k, sc_stream stream) {
  SC_REQUIRE(a != nullptr && b != nullptr && d != nullptr, "sc_selftest_umma: null argument");
  SC_TRY(umma_selftest(a, b, d, n, k, static_cast<cudaStream_t>(stream)));
  return 0;
}

int sc_selftest_umma_ts(const float* a, const float* b, float* d, int32_t n, int32_t k, sc_stream stream) {
  SC_REQUIRE(a != nullptr && b != nullptr && d != nullptr, "sc_selftest_umma_ts: null argument");
  SC_TRY(umma_selftest_ts(a, b, d, n, k, static_cast<cudaStream_t>(stream)));
  return 0;
}

int sc_probe_tma_gather(const sc_complex* w, int32_t in_channels, int32_t out_channels, int64_t n_modes, int64_t* cycles_out,
                        sc_stream stream) {
  SC_REQUIRE(w != nullptr && cycles_out != nullptr, "sc_probe_tma_gather: null argument");
  SC_TRY(tma_gather_probe(reinterpret_cast<const float2*>(w), in_channels, out_channels, n_modes,
                          reinterpret_cast<long long*>(cycles_out), static_cast<cudaStream_t>(stream)));
  return 0;
}

const char* sc_last_error(void) { return t_error.c_str(); }
uint64_t sc_kernel_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
const char* sc_build_info(void) {
  return "libspectral_conv_b200 sm_100a nvcc " SC_STR(__CUDACC_VER_MAJOR__) "." SC_STR(__CUDACC_VER_MINOR__)
         " +rows-kernels"
      ;
}

}  // extern "C"
