// Host launchers of the small HBM-bound kernels around the GEMMs and the flow core (aux_kernels.cu).
#pragma once
#include "lfi_common.cuh"

namespace lfi {
namespace aux {

// dst[b][i][j] = src[b*sb + i*si + j*sj] for i < rows, j < cols; columns [cols, ld) are zero filled.
int gather2d(float *dst, int ld, const float *src, long sb, long si, long sj, int batch, int rows, int cols, cudaStream_t st);

// Folded cond_transform weight: WcF[k*D + d][enc_offe[m] + e] = Wc[k][d][enc_off[m] + e] (+ Wc[..][enc_off[m] + E + e]
// for GRU-encoded modalities, whose two output halves are identical, models.py:64).
int fold_wc(float *wcf, const float *wc, const Dims &d, const lfi_shape &s, cudaStream_t st);
// Gradient of the fold: both halves receive the folded gradient.  dwc += unfold(dwcf)
int unfold_wc_grad(float *dwc, const float *dwcf, const Dims &d, const lfi_shape &s, cudaStream_t st);

// out[j] += scale * sum_r A[r*ld + j]
int colsum(float *out, const float *A, int ld, int rows, int cols, float scale, cudaStream_t st);

// ActNorm2d forward / reverse on [B,C] (modules.py:45-80)
int actnorm(const float *x, const float *bias, const float *logs, float *y, int B, int C, int reverse, cudaStream_t st);
// nll bits (modules.py:207-212 + models.py:563-565)
int nll(const float *z, const float *logdet, float *out, int B, int C, cudaStream_t st);

// Sliding windows of a raw modality stream into rows m = t'*B + b:
//   dst[(s*M + m)*ld + c] (layout_steps = 1) or dst[m*ld + s*dim + c] (layout_steps = 0, "enc: none" flatten)
//   = mask[(t'*B+b)*hist + s] * x[b][t0 + t' - hist + off + s][c],   off = 1 (window ends at t) or 0 (p1_face)
int gather_windows(float *dst, int ld, int layout_steps, const float *x, const float *mask, int B, int T, int dim,
                   int hist, int off, int t0, int Tp, cudaStream_t st);

// One step of the windowed encoder GRU for all M windows (nn.GRU from zero state, models.py:63-64).
//   a_i = mask * xp[b][tau] + b_ih ; a_h = gh (or 0 at s == 0) + b_hh
struct EncStep {
  const float *xp;      // [B*T][3E]   x @ W_ih^T, no bias
  const float *gh;      // [M][3E]     h_prev @ W_hh^T (nullptr at s == 0)
  const float *b_ih, *b_hh;
  const float *mask;    // [Tp][B][hist] or nullptr
  const float *hprev;   // [M][E] or nullptr
  float *h;             // [M][E]
  float *gates, *ahn;   // [M][3E], [M][E] stash (nullable)
  float *cond; int cond_ld;  // final step: also written to cond[m*cond_ld + e] (nullable)
  void *h_hi, *h_lo;    // optional bf16 planes of h [M][E] (tensor-core modes: next step's GEMM operand, dW_hh operand)
  int s, hist, B, T, Tp, t0, E;
  int gates16;          // gates stash in 16-bit fixed point (lfi_common.cuh: q_unorm16 / q_snorm16)
};
int enc_gate_fwd(const EncStep &a, cudaStream_t st);

// Gate backward of one window step for all M windows, writing the gate gradients in the form the batched weight-gradient
// GEMMs consume (fp32, or bf16 planes in the tensor-core modes) and accumulating the bias gradients in-kernel:
//   dah [M][3E] = (da_r, da_u, da_n * r)   (h-side pre-activations: dW_hh, dh_prev, db_hh)
//   dan [M][E]  =  da_n                    (i-side n block: dW_ih rows [2E,3E), db_ih)
struct EncStepBwd2 {
  const float *gates, *ahn, *hprev;
  float *dh;
  const float *dh_extra; int dh_extra_ld;
  float *dah32, *dan32;                      // fp32 outputs (nullable)
  void *dah_hi, *dah_lo, *dan_hi, *dan_lo;   // bf16 plane outputs (nullable; lo nullable)
  float *gb_ih, *gb_hh;                      // [3E] bias gradients, accumulated
  int M, E;
  int gates16;                               // gates stash in 16-bit fixed point
};
// part != nullptr: bias gradients without atomics - every block adds its four sums (r, u, n, n*r blocks of E columns) into its
// own row of part [enc_gate_bwd2_part_rows(M, E)][4E] (zeroed by the caller; the blocks of one launch own distinct rows and the
// window steps are stream ordered) and gb_ih / gb_hh are not touched; one fixed-order column reduction finishes them.
int enc_gate_bwd2(const EncStepBwd2 &a, cudaStream_t st, float *part = nullptr);
int enc_gate_bwd2_part_rows(int M, int E);

// Adjoint of gather_windows (same arguments, src in the layout gather_windows writes): dx [B][T][dim] is written for every frame,
// dx[b][tau][c] = sum of mask * src over the (t', s) with tau = t0 + t' - hist + off + s, zero where no window reads the frame.
// add != nullptr: [Tp][B][dim], add[t'][b][c] joins the sum of frame tau = t0 + t' as its last term (p1_face: the gradient of the
// flow input), so each element stays one thread's fixed-order sum
int window_grad(float *dx, const float *src, int ld, int layout_steps, const float *mask, int B, int T, int dim, int hist, int off, int t0,
                int Tp, cudaStream_t st, const float *add = nullptr);

// LU parametrisation helpers (modules.py:163-177)
int lu_build(float *Lm, float *Um, const float *l, const float *u, const float *log_s, const float *sign_s, int K, int C, cudaStream_t st);
int tri_inverse_f64(float *Linv, float *Uinv, double *scratch, const float *Lm, const float *Um, int K, int C, cudaStream_t st);
int lu_mask_grads(float *dl, float *du, float *dlog_s, const float *dL, const float *dU, const float *log_s,
                  const float *sign_s, int K, int C, cudaStream_t st);

// clip_grad_norm_ + Adam over a flat buffer (lets_face_it_glow.py:61-72)
int sumsq(float *out2, const float *g, size_t n, cudaStream_t st);
int clip_adam(float *theta, const float *grad, float *m, float *v, size_t n, float lr, float b1, float b2, float eps,
              float max_norm, float grad_scale, int step, const float *sumsq_in, cudaStream_t st, const float *hyper = nullptr);
// clip_grad_norm_ + torch.optim.SGD / RMSprop over a flat buffer, per-step scalars read from hyper (lfi_clip_sgd_dev /
// lfi_clip_rmsprop_dev give the layouts); buf, grad_avg nullptr = no momentum / not centered
int clip_sgd(float *theta, const float *grad, float *buf, size_t n, const float *hyper, float momentum, float dampening,
             float weight_decay, int nesterov, float max_norm, float grad_scale, const float *sumsq_in, cudaStream_t st);
int clip_rmsprop(float *theta, const float *grad, float *square_avg, float *grad_avg, float *buf, size_t n, const float *hyper,
                 float alpha, float eps, float weight_decay, float momentum, float max_norm, float grad_scale, const float *sumsq_in,
                 cudaStream_t st);

int fill(float *p, float v, size_t n, cudaStream_t st);

// masked window inputs straight into split-bf16 operand planes [hist][M][ldp] (ldp = round_up(dim, 8), padding zero): the
// gather_windows(layout_steps = 1) + split_to_planes pair in one pass (encoder weight-gradient operand)
int gather_windows_planes(void *hi, void *lo, int ldp, const float *x, const float *mask, int B, int T, int dim, int hist, int off, int t0,
                          int Tp, cudaStream_t st);
// out1[b*so + j] (+ out2[..] where (j % period) < lim2) += sum over rows of (hi + lo)[b][r][col0 + j]: column sums of split-bf16 planes
int colsum_planes(float *out1, float *out2, int period, int lim2, long so, const void *hi, const void *lo, int ld, long sb, int batch, int rows,
                  int col0, int cols, cudaStream_t st);
int expand_faces(const float *x, const float *means, const float *stds, size_t rows, int exp_dim, int jaw_dim, int neck_dim, float *out,
                 cudaStream_t st);
// calc_jerk (glow/utils.py:53-58): mean |third time difference| of x [B, T, C]; scratch: one double; out: one float
int jerk(const float *x, int B, int T, int C, double *scratch, float *out, cudaStream_t st);
// out[b][t][:] = raw[row0[b] + t][:]: a batch of stride-1 windows out of an HBM-resident corpus (mimicry_data_module.py:44-78)
int gather_batch(const float *raw, const long long *row0, int B, int T, int dim, float *out, cudaStream_t st);
}  // namespace aux
}  // namespace lfi
