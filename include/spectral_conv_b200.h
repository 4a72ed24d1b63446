/*
 * spectral_conv_b200.h -- C ABI of the B200-native SpectralConv hot path (libspectral_conv_b200.so).
 *
 * Drop-in boundary for ONE reference method and the backward PyTorch records for it:
 *
 *     neuralop/layers/spectral_convolution.py:417-570   SpectralConv.forward (real data, full precision)
 *
 * Plain pointers and sizes only: no torch / pybind types cross this boundary.  All `float*` / `sc_complex*`
 * arguments are DEVICE pointers on the device that was current when the plan was created; the caller
 * (neuraloperator_b200/spectral_conv.py on the Python side) owns every buffer, allocates outputs and
 * workspace through its own allocator (torch's caching allocator) and passes the CUDA stream to launch on.
 * Every entry point returns 0 on success, non-zero on failure (sc_last_error() describes it); there is
 * no CPU fallback behind any of them.
 *
 * Layouts (all contiguous, row-major):
 *   x, dx      float  (B, Ci, N_1..N_d)            input / its gradient; IEEE half or bfloat16 instead when the plan
 *                                                  carries SC_FLAG_GRID_F16 / SC_FLAG_GRID_BF16 (the `float*` arguments
 *                                                  then address 16-bit data)
 *   y, gy      float  (B, Co, M_1..M_d)            output / upstream gradient (M = N unless resampled)
 *   modes      sc_complex (B, C, k_1..k_d)         kept-mode block, ordered exactly like the reference's
 *                                                  x[slices_x] (:500-519): leading dims by increasing signed
 *                                                  frequency, last dim bins 0..k_d-1
 *   weight     sc_complex (Ci, Co, max_1..max_d)   dense weight as stored by the module (:354-369)
 *   bias       float  (Co)                         bias (Co,1,..,1) flattened (:376-379)
 */
#ifndef SPECTRAL_CONV_B200_H
#define SPECTRAL_CONV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SC_MAX_DIMS 4

typedef struct { float re, im; } sc_complex;   /* bit-compatible with torch.complex64 / cuFloatComplex */
typedef struct sc_plan sc_plan;                /* opaque; owns the device-resident twiddle tables */
typedef void* sc_stream;                       /* cudaStream_t */
typedef void* sc_event;                        /* cudaEvent_t */

enum { SC_NORM_FORWARD = 0, SC_NORM_BACKWARD = 1, SC_NORM_ORTHO = 2 };   /* fft_norm, :303,:342 */

/* What SpectralConv.forward derives from its arguments before touching data (:429-434, :465-528). */
typedef struct {
  int32_t ndim;                       /* 1..4 spatial dims ("order", :318)                                   */
  int32_t grid[SC_MAX_DIMS];          /* N_j : x.shape[2:]                                                   */
  int32_t out_grid[SC_MAX_DIMS];      /* M_j : output_shape / round(N_j * resolution_scaling_factor) (:524-528) */
  int32_t n_modes[SC_MAX_DIMS];       /* SpectralConv.n_modes as STORED (last already n//2+1, :404-415)       */
  int32_t max_n_modes[SC_MAX_DIMS];   /* SpectralConv.max_n_modes = weight extents along the mode dims (:317-321) */
  int32_t fft_norm;                   /* SC_NORM_*                                                           */
  int32_t flags;                      /* SC_FLAG_* (0 for SpectralConv.forward on float32 x)                 */
} sc_problem;
/* SC_FLAG_RESAMPLE: the synthesis places every kept SIGNED frequency f of a leading dim at bin (f mod M) of the output grid,
 * as neuralop/layers/resample.py:57-68 copies the spectrum corners (out_fft[..., -m//2:] = X[..., -m//2:]); without the flag
 * the unshifted spectrum is cropped / zero-padded at its end, as `ifftn(out_fft, s=...)` does in SpectralConv.forward (:548). */
enum { SC_FLAG_RESAMPLE = 1 };
/* SC_FLAG_GRID_F16 / SC_FLAG_GRID_BF16: the images on `grid` -- x, read by the forward analysis, and dx, written by the adjoint
 * synthesis -- are stored as IEEE half / bfloat16 (what a model trained under torch.autocast feeds the conv).  Images on `out_grid`
 * (y, gy) stay float.  The transforms compute in fp32 on the widened input, which every 16-bit value is exactly, so y equals the
 * result for x converted to float bit for bit; dx is the fp32 adjoint rounded to nearest even.  The two flags exclude each other and
 * SC_FLAG_RESAMPLE (sc_plan_create rejects those combinations before it touches a device); the tables do not depend on them, and
 * the workspace sizes grow by one fp32 copy of the images on `grid`. */
enum { SC_FLAG_GRID_F16 = 2, SC_FLAG_GRID_BF16 = 4 };

/* ---- plan: kept-mode index set + twiddle tables (replaces the slices built at :465-519) ---------------- */
int  sc_plan_create(const sc_problem* problem, sc_plan** plan_out);
void sc_plan_destroy(sc_plan* plan);
/* kept modes per dim k'_j = min(F_j, n_modes_j) (:466); returns ndim */
int  sc_plan_kept_modes(const sc_plan* plan, int32_t* kept_out);
/* unshifted spectrum bin read by kept slot t of dim `dim`, and the weight row it is multiplied with
 * (the content of slices_x after undoing fftshift, and of slices_w; :476-519).  Each array has kept[dim] entries. */
int  sc_plan_mode_bins(const sc_plan* plan, int dim, int32_t* in_bins_out, int32_t* weight_rows_out);
/* The same index set straight from a problem description: pure host arithmetic, needs no device (what the CPU tests compare
 * bit-exactly with the reference's slices).  kept_out: k'_dim; the two arrays must hold min(F_dim, n_modes_dim) entries. */
int  sc_problem_mode_bins(const sc_problem* problem, int dim, int32_t* kept_out, int32_t* in_bins_out,
                          int32_t* weight_rows_out);
/* The twiddle tables a plan for `problem` would upload, computed on the host (no device needed): the truncated transforms ARE
 * products with these tables, so applying them in numpy reproduces the library's arithmetic up to summation order -- this is how
 * the CPU tests check norms, the Hermitian rules of the C2R step (:552-559), resampling and odd sizes against the reference.
 * Row-major float32; complex tables are interleaved (re, im) and `cols_out` counts floats.  `out` may be NULL to query the shape.
 *   LAST_ANALYSIS          [N_d x 2k_d]   x-row -> (re, im) of the kept bins of the last dim, forward scale folded in
 *   LAST_SYNTHESIS         [2k_d x M_d]   (re, im) of the kept bins -> output row, C2R rules + inverse scale folded in
 *   LEAD_ANALYSIS (dim)    [k_j x N_j]    complex,  exp(-2 pi i b n / N_j) for the kept bins b in kept-slot order
 *   LEAD_SYNTHESIS (dim)   [M_j x k_j]    complex,  exp(+2 pi i b n / M_j) * [b < M_j]
 *   *_ADJOINT                             the conjugate transposes the backward pass multiplies with */
enum { SC_TABLE_LAST_ANALYSIS = 0, SC_TABLE_LAST_ANALYSIS_ADJOINT = 1, SC_TABLE_LAST_SYNTHESIS = 2,
       SC_TABLE_LAST_SYNTHESIS_ADJOINT = 3, SC_TABLE_LEAD_ANALYSIS = 4, SC_TABLE_LEAD_ANALYSIS_ADJOINT = 5,
       SC_TABLE_LEAD_SYNTHESIS = 6, SC_TABLE_LEAD_SYNTHESIS_ADJOINT = 7 };
int  sc_problem_table(const sc_problem* problem, int which, int dim, float* out, size_t out_capacity_floats,
                      int64_t* rows_out, int64_t* cols_out);
/* scratch the transform entry points need for `batch_times_channels` images (max over Ci, Co) */
size_t sc_workspace_bytes(const sc_plan* plan, int64_t batch_times_channels);
/* 0 = generic SIMT kernels only, 1 = tcgen05/TMA fused path where the shape qualifies (default) */
int  sc_plan_set_fast_path(sc_plan* plan, int enable);
int  sc_plan_uses_fast_path(const sc_plan* plan);
/* The persistent transform kernels launch one CTA per SM; the dx synthesis of sc_backward_dense, when called with a grads_ready
 * event, leaves n_sms of them free (default 0) so that the collective the caller runs on another stream (the data-parallel
 * gradient all-reduce) finds room for its own CTAs. */
int  sc_plan_set_reserved_sms(sc_plan* plan, int n_sms);

/* ---- the two transforms ------------------------------------------------------------------------------- */
/* Truncated analysis:  images (n_images, grid..) real  ->  modes (n_images, k_1..k_d).
 *   adjoint == 0 : rfftn(norm) + fftshift + x[slices_x]                      (:443-449, :500-519)  on `grid`
 *   adjoint == 1 : the adjoint of sc_synthesize (what autograd applies to gy): images live on `out_grid`.   */
int sc_analyze(const sc_plan* plan, const float* images, int64_t n_images, sc_complex* modes_out,
               int adjoint, void* workspace, size_t workspace_bytes, sc_stream stream);
/* Zero-padded synthesis: modes (n_images, k_1..k_d) -> images real.
 *   adjoint == 0 : scatter + ifftshift + ifftn(leading) + Hermitian fix + irfft(last) + bias   (:460-462,:520-568)
 *                  onto `out_grid`; bias (n_channels) may be NULL; image n uses bias[n % n_channels].
 *   adjoint == 1 : the adjoint of sc_analyze (produces dx on `grid`); bias must be NULL.                    */
int sc_synthesize(const sc_plan* plan, const sc_complex* modes_in, int64_t n_images, int32_t n_channels,
                  const float* bias, float* images_out, int adjoint,
                  void* workspace, size_t workspace_bytes, sc_stream stream);

/* ---- dense mode-wise contraction (_contract_dense, :21-46) and its backward ------------------------------ */
/* ym[b,o,m] = sum_i xm[b,i,m] * weight[i,o,w(m)] */
int sc_contract_dense(const sc_plan* plan, const sc_complex* xm, const sc_complex* weight, sc_complex* ym,
                      int32_t batch, int32_t in_channels, int32_t out_channels, sc_stream stream);
/* dxm[b,i,m] = sum_o gm[b,o,m] * conj(weight[i,o,w(m)])                 (dxm may be NULL)
 * dweight[i,o,w(m)] = sum_b conj(xm[b,i,m]) * gm[b,o,m], zero elsewhere  (dweight may be NULL; full weight shape)
 * dbias[o] = sum_{b,n} gy[b,o,n], read off the DC slot of gm             (dbias may be NULL) */
int sc_contract_dense_backward(const sc_plan* plan, const sc_complex* xm, const sc_complex* gm,
                               const sc_complex* weight, sc_complex* dxm, sc_complex* dweight, float* dbias,
                               int32_t batch, int32_t in_channels, int32_t out_channels, sc_stream stream);
/* dbias alone (used by the factorized paths): dbias[o] = sum_b Re(gm[b,o,DC]) / synthesis scale */
int sc_bias_grad(const sc_plan* plan, const sc_complex* gm, float* dbias, int32_t batch, int32_t out_channels,
                 sc_stream stream);

/* ---- building blocks of the factorized (Tucker) contraction, _contract_tucker :76-103, and of its backward --------- */
/* out[o, p, i] = sum_q op(table[p, q]) * in[o, q, i]   (complex; table element (p,q) at table[p*stride_p + q*stride_q];
 * op = conj when conj_table != 0).  Applies one factor matrix along one axis of a tensor: channel mixing with U_in / U_out
 * (i = flattened modes) and the expansion of the core along a mode axis with the (kept rows of the) mode factors. */
int sc_table_contract(const sc_complex* table, int64_t table_stride_p, int64_t table_stride_q, int conj_table,
                      const sc_complex* in, sc_complex* out, int64_t n_outer, int32_t P, int32_t Q, int32_t n_inner,
                      sc_stream stream);
/* out[p*out_stride_p + q*out_stride_q] = sum_{o, i} conj(a[o, p, i]) * b[o, q, i]   (a: [n_outer x P x n_inner],
 * b: [n_outer x Q x n_inner]): gradient of a factor matrix in PyTorch's conjugate convention (warp-shuffle reductions). */
int sc_pair_reduce(const sc_complex* a, const sc_complex* b, sc_complex* out, int64_t out_stride_p, int64_t out_stride_q,
                   int64_t n_outer, int32_t P, int32_t Q, int32_t n_inner, sc_stream stream);

/* ---- building blocks of the CP contraction, _contract_cp :55-73: out = U_out ( (x U_in) * scale ),  -------------------
 *      scale[e, m] = lambda[e] * prod_j U_j[m_j, e]  (mode_factors[j]: kept rows of factor j, [kept[j] x rank] row-major) */
int sc_cp_scale(const sc_complex* const* mode_factors, const int32_t* kept, int32_t ndim, const sc_complex* lambda,
                sc_complex* scale, int32_t rank, sc_stream stream);
/* out[a, e, m] = in[a, e, m] * op(scale[e, m])  (per_batch = rank * n_modes).  With e = channel and scale = the kept block of
 * a (C, modes..) weight this is also the separable contraction, _contract_dense_separable :49-52 (conj_scale = 1: its dxm). */
int sc_cp_apply(const sc_complex* in, const sc_complex* scale, sc_complex* out, int conj_scale, int32_t batch,
                int64_t per_batch, sc_stream stream);
/* dscale[e, m] = sum_a conj(t[a, e, m]) * g[a, e, m]   (separable: the weight gradient) */
int sc_cp_dscale(const sc_complex* t, const sc_complex* g, sc_complex* dscale, int32_t batch, int64_t per_batch,
                 sc_stream stream);
/* gradient of lambda (which = -1, out[rank]) or of mode factor `which` (out[kept[which] x rank]) from dscale */
int sc_cp_factor_grad(const sc_complex* const* mode_factors, const int32_t* kept, int32_t ndim, const sc_complex* lambda,
                      const sc_complex* dscale, sc_complex* out, int32_t which, int32_t rank, sc_stream stream);

/* ---- whole forward / backward for a dense weight (one call per autograd.Function.forward/backward) ------ */
/* y = SpectralConv.forward(x); xm_saved (B*Ci*prod(k) sc_complex, 32-byte aligned) is the only activation kept for backward.
 * It is OPAQUE: *saved_layout_out tells sc_backward_dense how its elements are ordered -- SC_MODES_STANDARD (B, Ci, k_1..k_d),
 * or SC_MODES_QUAD_MAJOR [prod(k)/4][B][Ci][4], which the fused tcgen05 chain uses so that the operand sectors of the
 * contraction kernels are contiguous.  Pass NULL to force the standard layout. */
enum { SC_MODES_STANDARD = 0, SC_MODES_QUAD_MAJOR = 1 };
int sc_forward_dense(const sc_plan* plan, const float* x, const sc_complex* weight, const float* bias,
                     float* y, sc_complex* xm_saved, int32_t* saved_layout_out,
                     int32_t batch, int32_t in_channels, int32_t out_channels,
                     void* workspace, size_t workspace_bytes, sc_stream stream);
/* saved_layout: what sc_forward_dense reported for xm_saved.  dx / dweight / dbias may each be NULL.
 * grads_ready (may be NULL): recorded on `stream` as soon as dweight and dbias are complete, i.e. BEFORE the dxm product and the
 * dx synthesis are launched: a data-parallel caller makes its collective stream wait on it and all-reduces the gradients
 * underneath the rest of the backward pass (DDP overlap, neuralop/training/trainer.py:203-205). */
int sc_backward_dense(const sc_plan* plan, const float* gy, const sc_complex* weight, const sc_complex* xm_saved,
                      int32_t saved_layout, float* dx, sc_complex* dweight, float* dbias,
                      int32_t batch, int32_t in_channels, int32_t out_channels,
                      void* workspace, size_t workspace_bytes, sc_stream stream, sc_event grads_ready);

/* ---- whole forward / backward for a Tucker weight, contracted factor by factor (_contract_tucker, :76-103) ----------------
 * ranks = {r_in, r_out, r_1..r_d} (the core's extents); core (r_in, r_out, r_1..r_d); u_in (Ci, r_in); u_out (Co, r_out);
 * u_modes[j] = the KEPT rows of mode factor j, contiguous (k_j, r_j) (`weight[slices_w]` slices the factors, :489).
 * plan_kept: the same problem with max_n_modes == kept modes (may be `plan` itself when nothing is cut).
 * `saved` (sc_tucker_saved_elems() elements, opaque) carries the activations backward needs: the kept input modes, the two
 * rank-channel intermediates, the expanded core and the expansion chain.  One workspace size serves both calls. */
size_t sc_tucker_saved_elems(const sc_plan* plan, int32_t batch, int32_t in_channels, int32_t out_channels, const int32_t* ranks);
size_t sc_tucker_workspace_bytes(const sc_plan* plan, int32_t batch, int32_t in_channels, int32_t out_channels, const int32_t* ranks);
int sc_forward_tucker(const sc_plan* plan, const sc_plan* plan_kept, const float* x, const sc_complex* core, const sc_complex* u_in,
                      const sc_complex* u_out, const sc_complex* const* u_modes, const float* bias, float* y, sc_complex* saved,
                      int32_t batch, int32_t in_channels, int32_t out_channels, const int32_t* ranks,
                      void* workspace, size_t workspace_bytes, sc_stream stream);
/* every gradient in the layout of its parameter (PyTorch conjugate convention); dbias may be NULL */
int sc_backward_tucker(const sc_plan* plan, const sc_plan* plan_kept, const float* gy, const sc_complex* core, const sc_complex* u_in,
                       const sc_complex* u_out, const sc_complex* const* u_modes, const sc_complex* saved, float* dx,
                       sc_complex* d_core, sc_complex* d_u_in, sc_complex* d_u_out, sc_complex* const* d_u_modes, float* dbias,
                       int32_t batch, int32_t in_channels, int32_t out_channels, const int32_t* ranks,
                       void* workspace, size_t workspace_bytes, sc_stream stream);

/* ---- whole forward / backward for a CP weight (_contract_cp, :55-73) and a TT weight (_contract_tt, :106-127), one call each ------
 * The launches of the per-factor building blocks above, in the same order and with the same operands as the Python-orchestrated
 * chains, issued from one opaque `saved` buffer and one workspace (graph-capturable, no host allocations in between).
 * CP: lambda (R), u_in (Ci, R), u_out (Co, R), u_modes[j] = the KEPT rows of mode factor j, contiguous (k_j, R).
 * TT: ranks = {r1, r_0 .. r_{d-1}}: g0 (1, Ci, r1), g1 (r1, Co, r_0), cores[j] = the KEPT rows of mode core j, contiguous
 *     (r_j, k_j, r_{j+1}) with r_d = 1; plan_kept as for the Tucker entry points.  Gradients in the layout of their parameter. */
size_t sc_cp_saved_elems(const sc_plan* plan, int32_t batch, int32_t in_channels, int32_t out_channels, int32_t rank);
size_t sc_cp_workspace_bytes(const sc_plan* plan, int32_t batch, int32_t in_channels, int32_t out_channels, int32_t rank);
int sc_forward_cp(const sc_plan* plan, const float* x, const sc_complex* lambda, const sc_complex* u_in, const sc_complex* u_out,
                  const sc_complex* const* u_modes, const float* bias, float* y, sc_complex* saved, int32_t batch, int32_t in_channels,
                  int32_t out_channels, int32_t rank, void* workspace, size_t workspace_bytes, sc_stream stream);
int sc_backward_cp(const sc_plan* plan, const float* gy, const sc_complex* lambda, const sc_complex* u_in, const sc_complex* u_out,
                   const sc_complex* const* u_modes, const sc_complex* saved, float* dx, sc_complex* d_lambda, sc_complex* d_u_in,
                   sc_complex* d_u_out, sc_complex* const* d_u_modes, float* dbias, int32_t batch, int32_t in_channels,
                   int32_t out_channels, int32_t rank, void* workspace, size_t workspace_bytes, sc_stream stream);
size_t sc_tt_saved_elems(const sc_plan* plan, int32_t batch, int32_t in_channels, int32_t out_channels, const int32_t* ranks);
size_t sc_tt_workspace_bytes(const sc_plan* plan, int32_t batch, int32_t in_channels, int32_t out_channels, const int32_t* ranks);
int sc_forward_tt(const sc_plan* plan, const sc_plan* plan_kept, const float* x, const sc_complex* g0, const sc_complex* g1,
                  const sc_complex* const* cores, const float* bias, float* y, sc_complex* saved, int32_t batch, int32_t in_channels,
                  int32_t out_channels, const int32_t* ranks, void* workspace, size_t workspace_bytes, sc_stream stream);
int sc_backward_tt(const sc_plan* plan, const sc_plan* plan_kept, const float* gy, const sc_complex* g0, const sc_complex* g1,
                   const sc_complex* const* cores, const sc_complex* saved, float* dx, sc_complex* d_g0, sc_complex* d_g1,
                   sc_complex* const* d_cores, float* dbias, int32_t batch, int32_t in_channels, int32_t out_channels, const int32_t* ranks,
                   void* workspace, size_t workspace_bytes, sc_stream stream);

/* ---- the one collective of the data-parallel step, over NVLink peer memory -------------------------------------------------
 * In-place all-reduce of `n_floats` (multiple of 4) floats: result = scale * sum over ranks (scale = 1 / world_size averages, as
 * DDP does, trainer.py:203-205).  peer_buffers[r] / peer_signal_pads[r] (HOST arrays of world_size DEVICE pointers) are rank r's
 * buffer and zero-initialised flag pad as mapped into THIS process -- CUDA symmetric memory (torch.distributed._symmetric_memory:
 * `rendezvous(...).buffer_ptrs / .signal_pad_ptrs`); the pad needs n_ctas * world_size 32-bit flags.  Every rank must call it with
 * the same n_floats / n_ctas; all n_ctas CTAs of a rank have to become resident together (they hand-shake with their peers), so keep
 * n_ctas at or below the SMs the concurrent kernels leave free (sc_plan_set_reserved_sms). */
int sc_allreduce_p2p(float* const* peer_buffers, uint32_t* const* peer_signal_pads, int32_t rank, int32_t world_size, int64_t n_floats,
                     float scale, int32_t n_ctas, sc_stream stream);

/* ---- Fourier-layer epilogue around the spectral convolution (SURVEY.md section 8, rows f1 / f2 / f3) ---------------------------
 * What neuralop/layers/fno_block.py:377-414 (`FNOBlocks.forward_with_postactivation`) does with the conv output, as ONE kernel
 * per channel-mixing step instead of one tensor pass per torch op.  Tensors are float (B, C, P) contiguous, P = points of the grid:
 *
 *   pre[b,o,p] = sum_i w[o*w_stride_o + i*w_stride_i] * in[b,i,p] + bias[o] + add[b,o,p] + gate[o] * gated[b,o,p]
 *   out        = act(pre)                      (SC_ACT_GELU = F.gelu's default exact erf form, fno_block.py:150)
 *
 *   f1  x1  = gelu( conv(x) + W_skip x )       in = x, w = fno_skips[i].conv.weight (Flattened1dConv, skip_connections.py:96-130),
 *                                              add = the SpectralConv output                                  (fno_block.py:379-397)
 *   f2  h   = gelu( W1 x1 + b1 )               ChannelMLP.fcs[0] (channel_mlp.py:63-116)
 *       out = act( W2 h + b2 + gate * x )      ChannelMLP.fcs[1] + SoftGating skip (skip_connections.py:53-93)  (fno_block.py:399-412)
 *
 * bias, add, gate, gated, pre_out may each be NULL (gate NULL with gated given = coefficient 1: the identity skip); in_channels may
 * be 0 (no mixing term: in / w unused).  pre_out (B, Co, P): the pre-activation, stored for the backward pass when given. */
enum { SC_ACT_IDENTITY = 0, SC_ACT_GELU = 1, SC_ACT_RELU = 2, SC_ACT_SILU = 3, SC_ACT_TANH = 4 };   /* non_linearity of the block */
int sc_channel_mix(const float* in, const float* w, int64_t w_stride_o, int64_t w_stride_i, const float* bias, const float* add,
                   const float* gate, const float* gated, int act, float* out, float* pre_out, int32_t batch, int32_t in_channels,
                   int32_t out_channels, int64_t n_points, sc_stream stream);
/* Backward, step 1 -- elementwise with the per-channel reductions folded in (pre may be NULL for SC_ACT_IDENTITY):
 *   gpre = gout * act'(pre)  -> gpre_out (may be NULL, may alias gout);  this is also the gradient of `add`
 *   dgated_out = gate[c] * gpre (may be NULL);  dbias[c] = sum_{b,p} gpre;  dgate[c] = sum_{b,p} gpre * gated  (each may be NULL)
 * Step 2, the gradient of `in`, is sc_channel_mix itself with the transposed weight strides (in = gpre, no adds, identity).
 * Step 3: dw[o, i] = sum_{b,p} gpre[b,o,p] * in[b,i,p]   (dw (Co, Ci) row-major = the layout of a Conv1d weight (Co, Ci, 1)). */
int sc_channel_mix_act_backward(const float* gout, const float* pre, int act, const float* gate, const float* gated, float* gpre_out,
                                float* dgated_out, float* dbias, float* dgate, int32_t batch, int32_t channels, int64_t n_points,
                                sc_stream stream);
int sc_channel_mix_weight_grad(const float* gpre, const float* in, float* dw, int32_t batch, int32_t in_channels, int32_t out_channels,
                               int64_t n_points, sc_stream stream);
/* sc_channel_mix on the tensor cores (tcgen05 bf16x3, activations as a tensor-memory A operand; Ci <= 256, Co <= 128): OPT-IN --
 * the kernel was written without hardware access, the exact-fp32 SIMT kernel stays the default.  Also enabled by SC_MIX_TC=1. */
int sc_layer_set_tensor_cores(int enable);
int sc_layer_uses_tensor_cores(void);
/* Elementwise helpers of the same layer: out[i] = op(a[i], b[i]).
 *   SC_POINTWISE_TANH           tanh(a)             the "tanh" stabilizer in front of the conv (fno_block.py:386-390)
 *   SC_POINTWISE_TANH_BACKWARD  a * (1 - b*b)       a = upstream gradient, b = tanh(x)
 *   SC_POINTWISE_ROUND_HALF     float(half(a))      the points where fno_block_precision "half" / "mixed" casts to fp16
 *                                                   (x.half() :436-437, x.chalf() :451-454, chalf output spectrum :456-462)
 *   SC_POINTWISE_ADD_I_TIMES    a + 1j * b          on interleaved complex (re, im) pairs: how `apply_complex` (neuralop/layers/complex.py:
 *                                                   55-62) combines the real and the imaginary module of a ComplexValued layer
 *   SC_POINTWISE_MUL_NEG_I      -1j * a             (the gradient of the above with respect to b); both: n even, out aliases no input
 *   SC_POINTWISE_MUL            a * b               dropout of the ChannelMLP (channel_mlp.py:54-58, 110-111): b = mask / (1 - p) */
enum { SC_POINTWISE_TANH = 0, SC_POINTWISE_TANH_BACKWARD = 1, SC_POINTWISE_ROUND_HALF = 2, SC_POINTWISE_ADD_I_TIMES = 3,
       SC_POINTWISE_MUL_NEG_I = 4, SC_POINTWISE_MUL = 5 };
int sc_pointwise(int op, const float* a, const float* b, float* out, int64_t n, sc_stream stream);
/* Host checks of the four kernels above: the kernels are sequences of __host__ __device__ tile functions; these entry points run
 * exactly those functions thread by thread, block by block, on HOST buffers (same arguments, no stream).  They exist so that the CPU
 * test tier can check the index arithmetic of the device code without a GPU; nothing in the Python package calls them. */
int sc_hostcheck_channel_mix(const float* in, const float* w, int64_t w_stride_o, int64_t w_stride_i, const float* bias, const float* add,
                             const float* gate, const float* gated, int act, float* out, float* pre_out, int32_t batch,
                             int32_t in_channels, int32_t out_channels, int64_t n_points);
int sc_hostcheck_channel_mix_act_backward(const float* gout, const float* pre, int act, const float* gate, const float* gated,
                                          float* gpre_out, float* dgated_out, float* dbias, float* dgate, int32_t batch,
                                          int32_t channels, int64_t n_points);
int sc_hostcheck_channel_mix_weight_grad(const float* gpre, const float* in, float* dw, int32_t batch, int32_t in_channels,
                                         int32_t out_channels, int64_t n_points);
int sc_hostcheck_pointwise(int op, const float* a, const float* b, float* out, int64_t n);
/* The element conversion of the 16-bit image storage (`flag` = SC_FLAG_GRID_F16 or SC_FLAG_GRID_BF16), run on the host through the
 * same __host__ __device__ pair the device kernels use.  to_16 == 0: n 16-bit values (uint16_t bit patterns) -> float; to_16 != 0:
 * n floats -> 16-bit, round to nearest even (overflow to +-inf, NaN stays NaN). */
int sc_hostcheck_convert(int flag, int to_16, const void* in, void* out, int64_t n);
/* Dry run of sc_forward_cp / sc_backward_cp (kind 0, ranks[0] = R) or sc_forward_tt / sc_backward_tt (kind 1) for `problem` on a
 * host-only plan: every primitive launch of the chain is RECORDED instead of executed -- {opcode, n_args, args...} words, pointers as
 * integers over synthetic buffer addresses (region << 40; regions listed at the definition in csrc/sc_api.cu) -- so that the CPU test
 * tier can replay the orchestration (which buffer goes where with which strides, in which order) on host arrays against the oracle.
 * log_out may be NULL to query the size; returns 0 and the word count in *n_words_out.  Test hook: the package never calls it. */
int sc_hostcheck_chain_log(const sc_problem* problem, int kind, int direction, int32_t batch, int32_t in_channels, int32_t out_channels,
                           const int32_t* ranks, int64_t* log_out, size_t capacity_words, int64_t* n_words_out);

/* events for the grads_ready hand-over above (timing disabled); sc_stream_wait_event makes `stream` wait for the last record */
int  sc_event_create(sc_event* event_out);
void sc_event_destroy(sc_event event);
int  sc_stream_wait_event(sc_stream stream, sc_event event);

/* ---- diagnostics --------------------------------------------------------------------------------------- */
const char* sc_last_error(void);          /* thread-local description of the last failure */
uint64_t    sc_kernel_launch_count(void); /* kernels this library has launched so far (process-wide) */
const char* sc_build_info(void);          /* "sm_100a nvcc <ver> ..." */
/* tcgen05 bring-up check: d[128 x n] = bf16(a[128 x k]) * bf16(b[n x k])^T accumulated in FP32 in TMEM, through the
 * same operand staging / descriptors / TMEM read-back the fused transform kernels use (device pointers, fp32). */
int sc_selftest_umma(const float* a, const float* b, float* d, int32_t n, int32_t k, sc_stream stream);
/* the same product with the A operand resident in tensor memory (tcgen05.st + TMEM-A tcgen05.mma) */
int sc_selftest_umma_ts(const float* a, const float* b, float* d, int32_t n, int32_t k, sc_stream stream);

/* measurement probe: one CTA per quad of modes gathers its (Ci x 64 x 32 B) block of a (Ci, 64, n_modes) complex64 tensor with 4-D
 * tensor loads; cycles_out[2q] = cycles to issue, cycles_out[2q+1] = cycles until every box has landed (device int64[2 * n_modes / 4]) */
int sc_probe_tma_gather(const sc_complex* w, int32_t in_channels, int32_t out_channels, int64_t n_modes, int64_t* cycles_out,
                        sc_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* SPECTRAL_CONV_B200_H */
