// Stand-alone module API under autograd: the backward passes of ActNorm2d / InvertibleConv1x1 / LinearZeros
// (modules.py:45-95, 122-194) and f_seq.forward with its backward (models.py:148-214), each on its own parameters; and the
// backward of FlowStep.forward in the reverse direction (FlowStep.reverse_flow, models.py:345-373) on one step of a flat
// parameter block.
//
// Every reduction over the B rows is deterministic: one CTA owns 32 columns and all rows of them, its 8 row groups sum in
// a fixed order and are combined in a fixed order (no atomics), and the weight-gradient GEMMs write their output tiles
// without split-K.  The same call twice therefore gives bit-identical gradients.  GEMMs run in LFI_GEMM_FP32, as the
// per-frame lfi_flowstep does.
#include "lfi_common.cuh"

namespace lfi {
const float *derived_winv(const Dims &d, const void *derived, int k);  // seq.cu

namespace {

// ---- column-reduction kernels -------------------------------------------------------------------
// For each column j of a [rows, cols] matrix d (pitch ld):
//   COL_SUM         s1[j] = sum_r d[r][j]
//   COL_ACTNORM     g = d e^{v[j]};   o = g;  s1[j] = sum g;   s2[j] = sum d * b            (b = y, the forward output)
//   COL_ACTNORM_REV g = d e^{-v[j]};  o = g;  s1[j] = -sum d;  s2[j] = -sum g * b          (b = x, the forward input)
//   COL_LINZ        g = d e^{f v[j]}; o = g;  s1[j] = sum g;   s2[j] = f * sum d * b       (b = out, the forward output)
enum { COL_SUM = 0, COL_ACTNORM = 1, COL_ACTNORM_REV = 2, COL_LINZ = 3 };
struct ColJob {
  const float *d, *b, *v;
  float *o, *s1, *s2;
  int rows, cols, ld;
  float f;
};
struct ColJobs {
  ColJob j[3];
};
constexpr int kColW = 32, kColRows = 8;

template <int MODE>
__global__ void __launch_bounds__(kColW * kColRows) colgrad_kernel(ColJobs jobs) {
  __shared__ float p1[kColRows][kColW + 1], p2[kColRows][kColW + 1];
  const ColJob &a = jobs.j[blockIdx.y];
  const int tx = threadIdx.x % kColW, ty = threadIdx.x / kColW;
  const int c = blockIdx.x * kColW + tx;
  if (blockIdx.x * kColW >= a.cols) return;  // whole CTA idle for this job (uniform across the block)
  float s1 = 0.f, s2 = 0.f;
  if (c < a.cols) {
    float e = 1.f;
    if (MODE == COL_ACTNORM) e = expf(a.v[c]);
    if (MODE == COL_ACTNORM_REV) e = expf(-a.v[c]);
    if (MODE == COL_LINZ) e = expf(a.f * a.v[c]);
    for (int r = ty; r < a.rows; r += kColRows) {
      const size_t i = (size_t)r * a.ld + c;
      const float d = a.d[i];
      if (MODE == COL_SUM) {
        s1 += d;
      } else {
        const float g = d * e;
        a.o[i] = g;
        if (MODE == COL_ACTNORM_REV) { s1 += d; s2 += g * a.b[i]; }
        else { s1 += g; s2 += d * a.b[i]; }
      }
    }
  }
  p1[ty][tx] = s1;
  p2[ty][tx] = s2;
  __syncthreads();
  if (ty == 0 && c < a.cols) {
#pragma unroll
    for (int i = 1; i < kColRows; ++i) { s1 += p1[i][tx]; s2 += p2[i][tx]; }
    if (MODE == COL_ACTNORM_REV) { s1 = -s1; s2 = -s2; }
    if (MODE == COL_LINZ) s2 *= a.f;
    a.s1[c] = s1;
    if (MODE != COL_SUM) a.s2[c] = s2;
  }
}

template <int MODE>
int launch_colgrad(const ColJobs &jobs, int njobs, cudaStream_t st) {
  int cmax = 0;
  for (int i = 0; i < njobs; ++i) cmax = jobs.j[i].cols > cmax ? jobs.j[i].cols : cmax;
  if (cmax <= 0) return LFI_OK;
  colgrad_kernel<MODE><<<dim3((cmax + kColW - 1) / kColW, njobs), kColW * kColRows, 0, st>>>(jobs);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

ColJob col_job(const float *d, int rows, int cols, int ld, float *s1) {
  ColJob j;
  memset(&j, 0, sizeof(j));
  j.d = d; j.rows = rows; j.cols = cols; j.ld = ld; j.s1 = s1;
  return j;
}

// ---- f_seq recurrent cell (torch.gru_cell / torch.lstm_cell) ------------------------------------
// gi = [z | c] W_ih^T + b_ih, gh = h W_hh^T + b_hh (gh == nullptr: zero state, gh = b_hh), both [B][G*H].
//   GRU  (r, u, n):    r = sig(gi_r + gh_r), u = sig(gi_u + gh_u), n = tanh(gi_n + r gh_n), h' = (1 - u) n + u h
//   LSTM (i, f, g, o): c' = sig(f) c + sig(i) tanh(g), h' = sig(o) tanh(c')
// Stash (all nullable): act [B][G*H] gate activations, ahn [B][H] = gh_n (GRU), h_st / c_st copies of h' / c'.
struct CellFwd {
  const float *gi, *gh, *b_hh, *h_prev, *c_prev;
  float *h_out, *c_out, *act, *ahn, *h_st, *c_st;
  int B, H, G;
};

__device__ __forceinline__ float sigm(float x) { return 1.0f / (1.0f + expf(-x)); }

__global__ void __launch_bounds__(256) cell_fwd_kernel(CellFwd a) {
  const size_t n = (size_t)a.B * a.H;
  const int GH = a.G * a.H;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const int b = (int)(e / a.H), j = (int)(e % a.H);
    const float *gi = a.gi + (size_t)b * GH;
    auto ah = [&](int q) { return a.gh ? a.gh[(size_t)b * GH + q * a.H + j] : a.b_hh[q * a.H + j]; };
    const float hp = a.h_prev ? a.h_prev[e] : 0.f;
    float *act = a.act ? a.act + (size_t)b * GH : nullptr;
    float h;
    if (a.G == 3) {
      const float hn = ah(2);
      const float r = sigm(gi[j] + ah(0));
      const float u = sigm(gi[a.H + j] + ah(1));
      const float nn = tanhf(gi[2 * a.H + j] + r * hn);
      h = (1.f - u) * nn + u * hp;
      if (act) { act[j] = r; act[a.H + j] = u; act[2 * a.H + j] = nn; }
      if (a.ahn) a.ahn[e] = hn;
    } else {
      const float cp = a.c_prev ? a.c_prev[e] : 0.f;
      const float ig = sigm(gi[j] + ah(0));
      const float fg = sigm(gi[a.H + j] + ah(1));
      const float gg = tanhf(gi[2 * a.H + j] + ah(2));
      const float og = sigm(gi[3 * a.H + j] + ah(3));
      const float c = fg * cp + ig * gg;
      h = og * tanhf(c);
      a.c_out[e] = c;
      if (a.c_st) a.c_st[e] = c;
      if (act) { act[j] = ig; act[a.H + j] = fg; act[2 * a.H + j] = gg; act[3 * a.H + j] = og; }
    }
    a.h_out[e] = h;
    if (a.h_st) a.h_st[e] = h;
  }
}

// Backward of one cell.  dh = dL/dh' from the LinearZeros product, plus dh_ext (nullable); dc_ext = dL/dc' (LSTM, nullable).
// Writes dai / dah [B][G*H] = dL/d(gi) / dL/d(gh) (equal except the GRU n block), dh_dir [B][H] = the direct part of
// dL/dh (u dh for the GRU, 0 for the LSTM; nullable) and dc_prev [B][H] = f dc (LSTM, nullable).
struct CellBwd {
  const float *act, *ahn, *c_st, *h_prev, *c_prev, *dh, *dh_ext, *dc_ext;
  float *dai, *dah, *dh_dir, *dc_prev;
  int B, H, G;
};

__global__ void __launch_bounds__(256) cell_bwd_kernel(CellBwd a) {
  const size_t n = (size_t)a.B * a.H;
  const int GH = a.G * a.H, H = a.H;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const int b = (int)(e / H), j = (int)(e % H);
    const float *act = a.act + (size_t)b * GH;
    float *dai = a.dai + (size_t)b * GH, *dah = a.dah + (size_t)b * GH;
    const float dh = a.dh[e] + (a.dh_ext ? a.dh_ext[e] : 0.f);
    const float hp = a.h_prev ? a.h_prev[e] : 0.f;
    if (a.G == 3) {
      const float r = act[j], u = act[H + j], nn = act[2 * H + j];
      const float dn = dh * (1.f - u) * (1.f - nn * nn);
      const float dr = dn * a.ahn[e] * r * (1.f - r);
      const float du = dh * (hp - nn) * u * (1.f - u);
      dai[j] = dr; dah[j] = dr;
      dai[H + j] = du; dah[H + j] = du;
      dai[2 * H + j] = dn; dah[2 * H + j] = dn * r;
      if (a.dh_dir) a.dh_dir[e] = dh * u;
    } else {
      const float ig = act[j], fg = act[H + j], gg = act[2 * H + j], og = act[3 * H + j];
      const float tc = tanhf(a.c_st[e]);
      const float cp = a.c_prev ? a.c_prev[e] : 0.f;
      const float dc = (a.dc_ext ? a.dc_ext[e] : 0.f) + dh * og * (1.f - tc * tc);
      const float d0 = dc * gg * ig * (1.f - ig), d1 = dc * cp * fg * (1.f - fg);
      const float d2 = dc * ig * (1.f - gg * gg), d3 = dh * tc * og * (1.f - og);
      dai[j] = d0; dai[H + j] = d1; dai[2 * H + j] = d2; dai[3 * H + j] = d3;
      dah[j] = d0; dah[H + j] = d1; dah[2 * H + j] = d2; dah[3 * H + j] = d3;
      if (a.dh_dir) a.dh_dir[e] = 0.f;
      if (a.dc_prev) a.dc_prev[e] = dc * fg;
    }
  }
}

// out[r][j] = o[r][j] * e^{f lf[j]} (torch: out * torch.exp(logs * logscale_factor)); copy: optional second destination
__global__ void __launch_bounds__(256) linz_scale_kernel(float *out, float *copy, const float *lf, float f, int rows, int cols) {
  const size_t n = (size_t)rows * cols;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const float v = out[e] * expf(f * lf[e % cols]);
    out[e] = v;
    if (copy) copy[e] = v;
  }
}

int grid_for(size_t n) {
  const size_t b = (n + 255) / 256;
  return (int)(b < 148 * 16 ? (b > 0 ? b : 1) : 148 * 16);
}

int gemm32(int tA, int tB, int M, int N, int K, const float *A, int lda, const float *Bm, int ldb, float *C, int ldc, int epi,
           const float *bias, cudaStream_t st, const float *aux = nullptr, int ldaux = 0) {
  GemmArgs g = gemm_args(tA, tB, M, N, K, A, lda, Bm, ldb, C, ldc, epi, bias);
  g.aux = aux; g.ldaux = ldaux;
  return gemm_dispatch(LFI_GEMM_FP32, g, nullptr, 0, st);
}

// ---- f_seq buffers ------------------------------------------------------------------------------
struct FseqDims {
  int In, Out, H, D, F, G, GH;
  float lf;
};
int fseq_dims(const lfi_fseq_shape *s, FseqDims *d) {
  LFI_REQUIRE(s, LFI_ERR_ARG, "f_seq: null shape");
  LFI_REQUIRE(s->In >= 1 && s->Out >= 1 && s->H >= 1 && s->D >= 1 && s->F >= 1, LFI_ERR_SHAPE,
              "f_seq: In=%d Out=%d H=%d D=%d F=%d must all be >= 1", s->In, s->Out, s->H, s->D, s->F);
  LFI_REQUIRE(s->G == 3 || s->G == 4, LFI_ERR_SHAPE, "f_seq: G=%d must be 3 (GRU) or 4 (LSTM)", s->G);
  d->In = s->In; d->Out = s->Out; d->H = s->H; d->D = s->D; d->F = s->F; d->G = s->G; d->GH = s->G * s->H;
  d->lf = s->logscale_factor;
  return LFI_OK;
}

struct FseqStash {  // caller-owned, opaque: activations of one f_seq.forward call on [B] rows
  float *cact, *act, *ahn, *h, *c, *out;
  size_t bytes;
};
void plan_fseq_stash(const FseqDims &d, int B, const void *base, FseqStash *s) {
  Bump b(const_cast<void *>(base), 0);
  s->cact = b.take<float>((size_t)B * d.D);
  s->act = b.take<float>((size_t)B * d.GH);
  s->ahn = b.take<float>((size_t)B * d.H);
  s->h = b.take<float>((size_t)B * d.H);
  s->c = b.take<float>((size_t)B * d.H);
  s->out = b.take<float>((size_t)B * d.Out);
  s->bytes = round_up_sz(b.off, 256);
}

struct FseqFwdWs {
  float *gi, *gh, *cact;
  size_t bytes;
};
void plan_fseq_fwd_ws(const FseqDims &d, int B, void *base, FseqFwdWs *w) {
  Bump b(base, 0);
  w->gi = b.take<float>((size_t)B * d.GH);
  w->gh = b.take<float>((size_t)B * d.GH);
  w->cact = b.take<float>((size_t)B * d.D);
  w->bytes = round_up_sz(b.off, 256);
}

struct FseqBwdWs {
  float *g, *dh, *dai, *dah, *dc;
  size_t bytes;
};
void plan_fseq_bwd_ws(const FseqDims &d, int B, void *base, FseqBwdWs *w) {
  Bump b(base, 0);
  w->g = b.take<float>((size_t)B * d.Out);
  w->dh = b.take<float>((size_t)B * d.H);
  w->dai = b.take<float>((size_t)B * d.GH);
  w->dah = b.take<float>((size_t)B * d.GH);
  w->dc = b.take<float>((size_t)B * d.D);
  w->bytes = round_up_sz(b.off, 256);
}

bool fseq_params_ok(const lfi_fseq_params *p) {
  return p && p->wc && p->bc && p->w_ih && p->b_ih && p->w_hh && p->b_hh && p->wf && p->bf && p->lf;
}

// Backward of f_seq on B rows (lfi_fseq_bwd, and the coupling network inside lfi_flowstep_rev_bwd), arguments checked by the
// caller.  z has row pitch z_ld; dz (nullable) has row pitch dz_ld and is written (dz_epi = 0) or added to (LFI_EPI_ACCUM_PRE:
// no split-K, unlike LFI_EPI_ACCUM).
int fseq_bwd_rows(const FseqDims &d, const lfi_fseq_params *p, const float *z, int z_ld, const float *cond, const float *h_in,
                  const float *c_in, const float *dout, const float *dh_out, const float *dc_out, float *dz, int dz_ld, int dz_epi,
                  float *dcond, float *dh_in, float *dc_in, lfi_fseq_params *g, int B, const FseqStash &q, const FseqBwdWs &w,
                  cudaStream_t st) {
  const int GH = d.GH, In = d.In, D = d.D, H = d.H, F = d.F, Out = d.Out, Wl = In + D;
  // LinearZeros: g = dout e^{f logs}, db_f, dlogs (one pass), dW_f = g^T h', dh' = g W_f
  ColJobs j;
  memset(&j, 0, sizeof(j));
  j.j[0] = col_job(dout, B, Out, Out, g->bf);
  j.j[0].b = q.out; j.j[0].v = p->lf; j.j[0].o = w.g; j.j[0].s2 = g->lf; j.j[0].f = d.lf;
  LFI_TRY(launch_colgrad<COL_LINZ>(j, 1, st));
  LFI_TRY(gemm32(1, 0, Out, H, B, w.g, Out, q.h, H, g->wf, H, 0, nullptr, st));
  LFI_TRY(gemm32(0, 0, B, H, Out, w.g, Out, p->wf, H, w.dh, H, 0, nullptr, st));
  // cell backward: gate gradients, the direct part of dh_in, dc_in
  CellBwd a;
  memset(&a, 0, sizeof(a));
  a.act = q.act; a.ahn = q.ahn; a.c_st = q.c; a.h_prev = h_in; a.c_prev = c_in; a.dh = w.dh; a.dh_ext = dh_out;
  a.dc_ext = d.G == 4 ? dc_out : nullptr; a.dai = w.dai; a.dah = w.dah; a.dh_dir = dh_in; a.dc_prev = d.G == 4 ? dc_in : nullptr;
  a.B = B; a.H = H; a.G = d.G;
  cell_bwd_kernel<<<grid_for((size_t)B * H), 256, 0, st>>>(a);
  LFI_LAUNCH_CHECK();
  if (dh_in) LFI_TRY(gemm32(0, 0, B, H, GH, w.dah, GH, p->w_hh, H, dh_in, H, LFI_EPI_ACCUM_PRE, nullptr, st));
  if (h_in) LFI_TRY(gemm32(1, 0, GH, H, B, w.dah, GH, h_in, H, g->w_hh, H, 0, nullptr, st));
  else LFI_CUDA(cudaMemsetAsync(g->w_hh, 0, (size_t)GH * H * sizeof(float), st));
  // gate-ih product over [z | c]: dW_ih in two column blocks, dz, and dc through LeakyReLU'
  LFI_TRY(gemm32(1, 0, GH, In, B, w.dai, GH, z, z_ld, g->w_ih, Wl, 0, nullptr, st));
  LFI_TRY(gemm32(1, 0, GH, D, B, w.dai, GH, q.cact, D, g->w_ih + In, Wl, 0, nullptr, st));
  if (dz) LFI_TRY(gemm32(0, 0, B, In, GH, w.dai, GH, p->w_ih, Wl, dz, dz_ld, dz_epi, nullptr, st));
  LFI_TRY(gemm32(0, 0, B, D, GH, w.dai, GH, p->w_ih + In, Wl, w.dc, D, LFI_EPI_LRELU_BWD, nullptr, st, q.cact, D));
  // bias gradients: db_ih = sum dai, db_hh = sum dah, db_c = sum dc (one launch)
  memset(&j, 0, sizeof(j));
  j.j[0] = col_job(w.dai, B, GH, GH, g->b_ih);
  j.j[1] = col_job(w.dah, B, GH, GH, g->b_hh);
  j.j[2] = col_job(w.dc, B, D, D, g->bc);
  LFI_TRY(launch_colgrad<COL_SUM>(j, 3, st));
  // cond_transform: dW_c = dc^T cond, dcond = dc W_c
  LFI_TRY(gemm32(1, 0, D, F, B, w.dc, D, cond, F, g->wc, F, 0, nullptr, st));
  if (dcond) LFI_TRY(gemm32(0, 0, B, F, D, w.dc, D, p->wc, F, dcond, F, 0, nullptr, st));
  return LFI_OK;
}

// ---- FlowStep.reverse_flow backward -------------------------------------------------------------
// Backward of the inverse coupling (models.py:358-366) on [B] rows, one thread per (row, channel pair q < Cz) that also
// passes column q < Ci through.  zc = [z1 | zc2] [B][C] and o [B][Co] (after its exp(3 logs) scale) come from the stash,
// dzc [B][C] = dL/dzc, dld [B] = dL/d(logdet) (nullable).
//   affine:   (shift, a) = (o[:, 0::2], o[:, 1::2]), s = max(sigmoid(a + 2), eps), zc2 = z2 / s - shift, ld -= sum log s
//   additive: zc2 = z2 - o
// z2 / s is recovered as zc2 + shift.  Writes dx [B][C] = (dL/dzc1, dL/dz2) - the f_seq path adds its dz1 to the first block
// later - and dO [B][Co] = dL/do (interleaved like o; the clamp passes the gradient where sigmoid(a + 2) >= eps, as torch's
// clamp does), and leaves dzc negated in place: the operand of dW = x1^T (-dzc).
__global__ void __launch_bounds__(256) coupling_rev_bwd_kernel(const float *zc, const float *o, float *dzc, const float *dld,
                                                                float *dx, float *dO, int B, int C, int Ci, int Co, int affine,
                                                                float eps) {
  const int Cz = C - Ci;
  const size_t n = (size_t)B * Cz;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const int b = (int)(e / Cz), q = (int)(e % Cz);
    const size_t r = (size_t)b * C;
    if (q < Ci) {
      const float g1 = dzc[r + q];
      dx[r + q] = g1;
      dzc[r + q] = -g1;
    }
    const float g = dzc[r + Ci + q];
    float *dOr = dO + (size_t)b * Co;
    if (affine) {
      const float shift = o[(size_t)b * Co + 2 * q], sg = sigm(o[(size_t)b * Co + 2 * q + 1] + 2.0f);
      const float s = fmaxf(sg, eps);
      const float ds = -(g * (zc[r + Ci + q] + shift) + (dld ? dld[b] : 0.f)) / s;
      dOr[2 * q] = -g;
      dOr[2 * q + 1] = sg >= eps ? ds * sg * (1.f - sg) : 0.f;
      dx[r + Ci + q] = g / s;
    } else {
      dOr[q] = -g;
      dx[r + Ci + q] = g;
    }
    dzc[r + Ci + q] = -g;
  }
}

struct RevBwdWs {
  float *dx1, *dzc, *dO;
  FseqBwdWs f;
  size_t bytes;
};
void plan_rev_bwd_ws(const Dims &d, const FseqDims &fd, int B, void *base, RevBwdWs *w) {
  Bump b(base, 0);
  w->dx1 = b.take<float>((size_t)B * d.C);
  w->dzc = b.take<float>((size_t)B * d.C);
  w->dO = b.take<float>((size_t)B * d.Co);
  const size_t off = round_up_sz(b.off, 256);
  plan_fseq_bwd_ws(fd, B, base ? (char *)base + off : nullptr, &w->f);
  w->bytes = off + w->f.bytes;
}

// f_seq of step k: its shape, and its parameters (or their gradients) inside a flat [K, ...] block
FseqDims step_fseq_dims(const Dims &d) {
  FseqDims f;
  f.In = d.Ci; f.Out = d.Co; f.H = d.H; f.D = d.D; f.F = d.F; f.G = d.G; f.GH = d.GH; f.lf = 3.0f;
  return f;
}
template <class P>
lfi_fseq_params step_fseq_params(const Dims &d, P *p, int k) {
  const size_t GH = d.GH, In = d.Ci + d.D;
  lfi_fseq_params f;
  f.wc = p->wc + (size_t)k * d.D * d.F; f.bc = p->bc + (size_t)k * d.D;
  f.w_ih = p->w_ih + k * GH * In; f.b_ih = p->b_ih + k * GH;
  f.w_hh = p->w_hh + k * GH * d.H; f.b_hh = p->b_hh + k * GH;
  f.wf = p->wf + (size_t)k * d.Co * d.H; f.bf = p->bf + (size_t)k * d.Co; f.lf = p->lf + (size_t)k * d.Co;
  return f;
}

}  // namespace

// Bias gradients of an encoder GRU from the per-block partial sums of aux::enc_gate_bwd2 (part [rows][4E]: r, u, n, n*r blocks of
// E columns): db_ih = (r, u, n), db_hh = (r, u, n*r), written; every column summed over the rows in a fixed order (one launch).
int enc_bias_grads(const float *part, int rows, int E, float *gb_ih, float *gb_hh, cudaStream_t st) {
  ColJobs j;
  memset(&j, 0, sizeof(j));
  j.j[0] = col_job(part, rows, 3 * E, 4 * E, gb_ih);
  j.j[1] = col_job(part, rows, 2 * E, 4 * E, gb_hh);
  j.j[2] = col_job(part + 3 * E, rows, E, 4 * E, gb_hh + 2 * E);
  return launch_colgrad<COL_SUM>(j, 3, st);
}

}  // namespace lfi

using namespace lfi;

extern "C" {

int lfi_actnorm_bwd(const float *x, const float *y, const float *logs, const float *dy, float *dx, float *dbias, float *dlogs, int B,
                    int C, int reverse, void *stream) {
  const float *saved = reverse ? x : y;
  LFI_REQUIRE(saved && logs && dy && dx && dbias && dlogs, LFI_ERR_ARG, "lfi_actnorm_bwd: null argument");
  LFI_REQUIRE(B >= 1 && C >= 1, LFI_ERR_SHAPE, "lfi_actnorm_bwd: B=%d C=%d", B, C);
  ColJobs j;
  memset(&j, 0, sizeof(j));
  j.j[0] = col_job(dy, B, C, C, dbias);
  j.j[0].b = saved; j.j[0].v = logs; j.j[0].o = dx; j.j[0].s2 = dlogs;
  cudaStream_t st = (cudaStream_t)stream;
  return reverse ? launch_colgrad<COL_ACTNORM_REV>(j, 1, st) : launch_colgrad<COL_ACTNORM>(j, 1, st);
}

size_t lfi_linear_zeros_bwd_ws_bytes(int B, int Out) {
  if (B < 1 || Out < 1) return 0;
  return round_up_sz((size_t)B * Out * sizeof(float), 256);
}

int lfi_linear_zeros_bwd(const float *h, const float *w, const float *logs, const float *out, const float *dout, float logscale_factor,
                         float *dh, float *dw, float *db, float *dlogs, int B, int In, int Out, void *ws, size_t ws_bytes, void *stream) {
  LFI_REQUIRE(h && w && logs && out && dout && dh && dw && db && dlogs && ws, LFI_ERR_ARG, "lfi_linear_zeros_bwd: null argument");
  LFI_REQUIRE(B >= 1 && In >= 1 && Out >= 1, LFI_ERR_SHAPE, "lfi_linear_zeros_bwd: B=%d In=%d Out=%d", B, In, Out);
  LFI_REQUIRE(ws_bytes >= lfi_linear_zeros_bwd_ws_bytes(B, Out), LFI_ERR_WORKSPACE, "lfi_linear_zeros_bwd: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  float *g = (float *)ws;
  ColJobs j;
  memset(&j, 0, sizeof(j));
  j.j[0] = col_job(dout, B, Out, Out, db);
  j.j[0].b = out; j.j[0].v = logs; j.j[0].o = g; j.j[0].s2 = dlogs; j.j[0].f = logscale_factor;
  LFI_TRY(launch_colgrad<COL_LINZ>(j, 1, st));
  LFI_TRY(gemm32(0, 0, B, In, Out, g, Out, w, In, dh, In, 0, nullptr, st));  // dh = g W
  return gemm32(1, 0, Out, In, B, g, Out, h, In, dw, In, 0, nullptr, st);    // dW = g^T h
}

size_t lfi_fseq_ws_bytes(const lfi_fseq_shape *s, int B) {
  FseqDims d;
  if (fseq_dims(s, &d) != LFI_OK || B < 1) return 0;
  FseqFwdWs w;
  plan_fseq_fwd_ws(d, B, nullptr, &w);
  return w.bytes;
}

size_t lfi_fseq_stash_bytes(const lfi_fseq_shape *s, int B) {
  FseqDims d;
  if (fseq_dims(s, &d) != LFI_OK || B < 1) return 0;
  FseqStash q;
  plan_fseq_stash(d, B, nullptr, &q);
  return q.bytes;
}

size_t lfi_fseq_bwd_ws_bytes(const lfi_fseq_shape *s, int B) {
  FseqDims d;
  if (fseq_dims(s, &d) != LFI_OK || B < 1) return 0;
  FseqBwdWs w;
  plan_fseq_bwd_ws(d, B, nullptr, &w);
  return w.bytes;
}

int lfi_fseq_fwd(const lfi_fseq_shape *s, const lfi_fseq_params *p, const float *z, const float *cond, const float *h_in,
                 const float *c_in, float *h_out, float *c_out, float *out, int B, void *stash, size_t stash_bytes, void *ws,
                 size_t ws_bytes, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  FseqDims d;
  LFI_TRY(fseq_dims(s, &d));
  LFI_REQUIRE(fseq_params_ok(p) && z && cond && h_out && out && ws, LFI_ERR_ARG, "lfi_fseq_fwd: null argument");
  LFI_REQUIRE(d.G == 3 || c_out, LFI_ERR_ARG, "lfi_fseq_fwd: LSTM needs c_out");
  LFI_REQUIRE(B >= 1, LFI_ERR_SHAPE, "lfi_fseq_fwd: B=%d", B);
  FseqFwdWs w;
  plan_fseq_fwd_ws(d, B, ws, &w);
  LFI_REQUIRE(ws_bytes >= w.bytes, LFI_ERR_WORKSPACE, "lfi_fseq_fwd: workspace too small: %zu < %zu", ws_bytes, w.bytes);
  FseqStash q;
  memset(&q, 0, sizeof(q));
  if (stash) {
    plan_fseq_stash(d, B, stash, &q);
    LFI_REQUIRE(stash_bytes >= q.bytes, LFI_ERR_WORKSPACE, "lfi_fseq_fwd: stash too small: %zu < %zu", stash_bytes, q.bytes);
  }
  float *cact = stash ? q.cact : w.cact;
  const int GH = d.GH, In = d.In, D = d.D, H = d.H, Wl = In + D;
  // c = LeakyReLU(cond W_c^T + b_c); gates_i = c W_ih[:, In:]^T + b_ih + z W_ih[:, :In]^T  ([z | c] without a concatenated copy)
  LFI_TRY(gemm32(0, 1, B, D, d.F, cond, d.F, p->wc, d.F, cact, D, LFI_EPI_BIAS | LFI_EPI_LRELU, p->bc, st));
  LFI_TRY(gemm32(0, 1, B, GH, D, cact, D, p->w_ih + In, Wl, w.gi, GH, LFI_EPI_BIAS, p->b_ih, st));
  LFI_TRY(gemm32(0, 1, B, GH, In, z, In, p->w_ih, Wl, w.gi, GH, LFI_EPI_ACCUM_PRE, nullptr, st));
  if (h_in) LFI_TRY(gemm32(0, 1, B, GH, H, h_in, H, p->w_hh, H, w.gh, GH, LFI_EPI_BIAS, p->b_hh, st));
  CellFwd a;
  memset(&a, 0, sizeof(a));
  a.gi = w.gi; a.gh = h_in ? w.gh : nullptr; a.b_hh = p->b_hh; a.h_prev = h_in; a.c_prev = c_in;
  a.h_out = h_out; a.c_out = c_out; a.B = B; a.H = H; a.G = d.G;
  if (stash) { a.act = q.act; a.ahn = d.G == 3 ? q.ahn : nullptr; a.h_st = q.h; a.c_st = d.G == 4 ? q.c : nullptr; }
  cell_fwd_kernel<<<grid_for((size_t)B * H), 256, 0, st>>>(a);
  LFI_LAUNCH_CHECK();
  // LinearZeros: (h' W_f^T + b_f) e^{f logs}
  LFI_TRY(gemm32(0, 1, B, d.Out, H, h_out, H, p->wf, H, out, d.Out, LFI_EPI_BIAS, p->bf, st));
  linz_scale_kernel<<<grid_for((size_t)B * d.Out), 256, 0, st>>>(out, stash ? q.out : nullptr, p->lf, d.lf, B, d.Out);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

int lfi_fseq_bwd(const lfi_fseq_shape *s, const lfi_fseq_params *p, const float *z, const float *cond, const float *h_in,
                 const float *c_in, const float *dout, const float *dh_out, const float *dc_out, float *dz, float *dcond, float *dh_in,
                 float *dc_in, lfi_fseq_params *g, int B, const void *stash, size_t stash_bytes, void *ws, size_t ws_bytes,
                 void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  FseqDims d;
  LFI_TRY(fseq_dims(s, &d));
  LFI_REQUIRE(fseq_params_ok(p) && fseq_params_ok(g) && z && cond && dout && stash && ws, LFI_ERR_ARG, "lfi_fseq_bwd: null argument");
  LFI_REQUIRE(B >= 1, LFI_ERR_SHAPE, "lfi_fseq_bwd: B=%d", B);
  FseqStash q;
  plan_fseq_stash(d, B, stash, &q);
  LFI_REQUIRE(stash_bytes >= q.bytes, LFI_ERR_WORKSPACE, "lfi_fseq_bwd: stash too small: %zu < %zu", stash_bytes, q.bytes);
  FseqBwdWs w;
  plan_fseq_bwd_ws(d, B, ws, &w);
  LFI_REQUIRE(ws_bytes >= w.bytes, LFI_ERR_WORKSPACE, "lfi_fseq_bwd: workspace too small: %zu < %zu", ws_bytes, w.bytes);
  return fseq_bwd_rows(d, p, z, d.In, cond, h_in, c_in, dout, dh_out, dc_out, dz, d.In, 0, dcond, dh_in, dc_in, g, B, q, w, st);
}

size_t lfi_flowstep_rev_bwd_ws_bytes(const lfi_shape *s, int B) {
  Dims d;
  if (make_dims(s, &d) != LFI_OK || B < 1) return 0;
  RevBwdWs w;
  plan_rev_bwd_ws(d, step_fseq_dims(d), B, nullptr, &w);
  return w.bytes;
}

int lfi_flowstep_rev_bwd(const lfi_shape *s, const void *derived, const lfi_params *p, int k, const float *cond, const float *h_in,
                         const float *c_in, const float *dy, const float *dlogdet, const float *dh_out, const float *dc_out, float *dx,
                         float *dcond, float *dh_in, float *dc_in, lfi_params *g, int B, void *stash, size_t stash_bytes, void *ws,
                         size_t ws_bytes, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  Dims d;
  LFI_TRY(make_dims(s, &d));
  LFI_REQUIRE(derived && p && cond && dy && dx && dcond && dh_in && g && stash && ws, LFI_ERR_ARG, "lfi_flowstep_rev_bwd: null argument");
  LFI_REQUIRE(p->an_logs && p->wc && p->bc && p->w_ih && p->b_ih && p->w_hh && p->b_hh && p->wf && p->bf && p->lf, LFI_ERR_ARG,
              "lfi_flowstep_rev_bwd: null parameter block");
  LFI_REQUIRE(g->an_bias && g->an_logs && g->w && g->wc && g->bc && g->w_ih && g->b_ih && g->w_hh && g->b_hh && g->wf && g->bf && g->lf,
              LFI_ERR_ARG, "lfi_flowstep_rev_bwd: null gradient block");
  LFI_REQUIRE(k >= 0 && k < d.K && B >= 1, LFI_ERR_ARG, "lfi_flowstep_rev_bwd: bad step %d / batch %d", k, B);
  LFI_REQUIRE(d.G == 3 || dc_in, LFI_ERR_ARG, "lfi_flowstep_rev_bwd: LSTM needs dc_in");
  StepStash q;
  plan_step_stash(d, B, stash, &q);
  LFI_REQUIRE(stash_bytes >= q.bytes, LFI_ERR_WORKSPACE, "flowstep stash too small: %zu < %zu", stash_bytes, q.bytes);
  const FseqDims fd = step_fseq_dims(d);
  RevBwdWs w;
  plan_rev_bwd_ws(d, fd, B, ws, &w);
  LFI_REQUIRE(ws_bytes >= w.bytes, LFI_ERR_WORKSPACE, "flowstep reverse backward workspace too small: %zu < %zu", ws_bytes, w.bytes);
  const int C = d.C;
  const size_t kC = (size_t)k * C;
  // 1. reverse ActNorm, out = x1 e^{-logs} - bias: dx1, d bias, d logs (one pass)
  ColJobs j;
  memset(&j, 0, sizeof(j));
  j.j[0] = col_job(dy, B, C, C, g->an_bias + kC);
  j.j[0].b = q.y; j.j[0].v = p->an_logs + kC; j.j[0].o = w.dx1; j.j[0].s2 = g->an_logs + kC;
  LFI_TRY(launch_colgrad<COL_ACTNORM_REV>(j, 1, st));
  // 2. inverse 1x1 conv, x1 = zc W^-1: dzc = dx1 W^-T
  LFI_TRY(gemm32(0, 1, B, C, C, w.dx1, C, derived_winv(d, derived, k), d.Cp, w.dzc, C, 0, nullptr, st));
  // 3. inverse coupling: dO, dL/dz2, the pass-through dL/dz1 (and -dzc for step 5)
  coupling_rev_bwd_kernel<<<grid_for((size_t)B * d.Cz), 256, 0, st>>>(q.zf, q.o, w.dzc, dlogdet, dx, w.dO, B, C, d.Ci, d.Co, d.affine,
                                                                      d.eps);
  LFI_LAUNCH_CHECK();
  // 4. f_seq on z1 = zc[:, :Ci] with step k's parameters; its dz1 is added to dx[:, :Ci]
  FseqStash fq;
  fq.cact = q.Cact; fq.act = q.gates; fq.ahn = q.ahn; fq.h = q.h; fq.c = q.c; fq.out = q.o; fq.bytes = q.bytes;
  const lfi_fseq_params fp = step_fseq_params(d, p, k);
  lfi_fseq_params fg = step_fseq_params(d, g, k);
  LFI_TRY(fseq_bwd_rows(fd, &fp, q.zf, C, cond, h_in, c_in, w.dO, dh_out, dc_out, dx, C, LFI_EPI_ACCUM_PRE, dcond, dh_in, dc_in, &fg, B,
                        fq, w.f, st));
  // 5. dW of the forward weight: with Winv = W^-1, dW = -W^-T (zc^T dx1) W^-T = -(zc W^-1)^T (dx1 W^-T) = x1^T (-dzc)
  return gemm32(1, 0, C, C, B, q.y, C, w.dzc, C, g->w + (size_t)k * C * C, C, 0, nullptr, st);
}

}  // extern "C"
