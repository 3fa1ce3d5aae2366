// Kernel argument blocks and host launchers of the sequential flow core.
#pragma once
#include "core_tile.cuh"

namespace lfi {
namespace core {

// Activation stash written by the forward wavefront and consumed by the backward one.
// Every array is [K][Tp][B][width] (cell-major), fp32.
struct Stash {
  float *y;      // [.,C]   ActNorm output (input of the 1x1 conv)
  float *zf;     // [.,C]   1x1 conv output (z1 | z2)
  float *h;      // [.,H]   RNN state after the cell
  float *c;      // [.,H]   LSTM cell state after the cell (G == 4)
  float *gates;  // [.,GH]  post-activation gates
  float *ahn;    // [.,H]   GRU: h-side pre-activation of the n gate
  float *o;      // [.,Co]  LinearZeros output
  float *xin;    // [.,C]   input of step k (k >= 1; slot k = K unused)
};

// tensor-core side of the hybrid wavefronts (zero = off)
struct WaveTc {
  int mode;                      // lfi_gemm_mode of the batched products (0 = off)
  const void *whh_hi, *whh_lo;   // bf16 planes of W_hh [K][GH][H] (lo null in bf16 mode), split once per call
  float *ghbuf;                  // [2][K][B][GH] products of two consecutive wavefronts (forward)
  void *gws; size_t gws_bytes;   // operand-plane scratch of the GEMMs
};

struct FwdArgs {
  Dims d;
  DerivedView dv;
  int B, Tp;
  int k_first, k_last;        // step range evaluated (module API: a single step)
  const float *x0;            // input of step k_first: element (b, t, c) at x0[b*x_sb + t*x_st + c]
  long x_sb, x_st;
  const float *G;             // [Tp*B][g_ld] gate-ih pre-activations incl. b_ih; columns (k - g_k0)*GH ...
  long g_ld; int g_k0;
  const float *h0, *c0;       // [K][B][H] or nullptr (zeros)
  float *xin;                 // handoff between steps
  float *st_y, *st_zf, *st_h, *st_c, *st_gates, *st_ahn, *st_o;
  float *ld;                  // [Tp][B] running log-det (coupling terms only)
  int ld_accumulate;          // 1: ld already holds the caller's log-det
  float *nll;                 // [Tp][B] or nullptr
  float *z_out;               // [Tp][B][C] output of step k_last
  float *scale_out;           // [K][B][Cz] or nullptr (FlowStep.scale, models.py:336-337)
  int *flags; size_t flags_bytes;  // progress counters of the stage-pipelined kernel (nullptr: wavefront kernels only)
  // tensor-core modes, stage-pipelined kernel only: bf16 operand planes (hi, lo = bf16(v - hi); lo nullable) of the stash
  // entries the weight-gradient GEMMs contract over, written next to the fp32 stash
  void *py_hi, *py_lo, *pzf_hi, *pzf_lo, *ph_hi, *ph_lo;
  // 1: st_gates / st_ahn / st_h use the tiled layout of the tensor-core pipeline (core_pipe.cuh: stash_tiled_off), which makes
  // the thread-per-sequence stores of that kernel contiguous; the backward pipeline reads the same layout
  int stash_tiled;
  int g_tiled;  // 1: G is row-interleaved (core_pipe.cuh: g_tiled_off with ld = g_ld), tensor-core pipeline only
  // Hybrid wavefronts (tensor-core GEMM modes, shapes the stage pipelines do not cover - e.g. the wide variant K = 32, H = 256,
  // LSTM): the recurrent product h[k][t-1] W_hh[k]^T of every cell of a wavefront is ONE batched tcgen05 GEMM issued before the
  // wavefront's launch (core_fwd.cu: launch_fwd_t), and the cell kernel adds the result instead of streaming W_hh through FFMA.
  WaveTc wtc;
  union {
    const float *gh_pre;      // hybrid wavefronts, set per wavefront by the launcher: [K][B][GH] products of this wavefront's cells (t >= 1)
    // stage pipelines, with h0: the carry instantiation (time-chunked evaluation, lfi_seq_eval) runs; every sequence starts from
    // h0 and its state after frame Tp - 1 goes to h_last [K][B][H], st_h is not written.  (Sharing gh_pre's storage keeps the
    // argument block's size, so the kernels without a carried state are unchanged; launch_fwd refuses h_last for the wavefronts.)
    float *h_last;
  };
};

struct InvArgs {
  Dims d;
  DerivedView dv;
  int B, Tc;                  // frames in this launch
  int k_hi, k_lo;             // steps evaluated per frame, k_hi down to k_lo (whole flow: K-1 .. 0)
  int g_k0;                   // step whose gate-ih pre-activations sit at column 0 of G
  int t_abs0;                 // absolute frame index (into faces) of the first generated frame
  int t_rel0;                 // index of that frame relative to start_ts (into noise / logdet_out)
  const float *noise;         // [T'][B][C] or nullptr (zeros)
  const float *G; long g_ld;  // teacher-forced: [Tc*B][K*GH] gate-ih pre-activations (chunk-relative rows)
  const float *cstatic; long cs_ld;  // AR: [Tc*B][K*D] static part of cond_transform pre-activation (incl. bias)
  const float *faces; long f_sb, f_st;        // AR window source (seed + generated frames)
  float *faces_out; long fo_sb, fo_st;        // where frame t_abs is written
  float *hstate, *cstate;     // [K][B][H] carried RNN state (in/out)
  float *logdet_out;          // [T'][B] or nullptr (coupling terms only)
  // Module API (lfi_flowstep_rev_fwd_train: ONE frame, ONE step): nullptr, or the step's activations for its backward, all
  // [B][width], in the conventions of the forward stash (core::Stash): x1 = zc W^-1 (input of the reverse ActNorm), zc (coupling
  // output, input of the inverse 1x1 conv), post-activation gates, ahn (GRU), o after its exp(3 logs) scale.  Set together; a
  // launch with st_x1 set runs the kernels' stash instantiation.
  float *st_x1, *st_zc, *st_gates, *st_ahn, *st_o;
};

struct BwdArgs {
  Dims d;
  DerivedView dv;
  int B, Tp;
  const float *dnll;          // [Tp][B] dL/dnll
  const float *z;             // [Tp][B][C] forward output (for d nll / d z)
  Stash st;
  float *dx;                  // [K][Tp][B][C]  grad wrt input of step k (handoff)
  float *dh;                  // [K][Tp][B][H]  grad wrt h[k][t-1] produced by cell (k,t)
  float *dc;                  // [K][Tp][B][H]  LSTM
  float *dG;                  // [Tp*B][K*GH]   dA_i (grad wrt gate-ih pre-activation)
  float *dAh;                 // [K][Tp][B][GH] dA_h (for dW_hh)
  float *dO;                  // [K][Tp][B][Co] grad wrt the LinearZeros matmul output (dO * exp(3 logs)), for dWf
  float *dzf;                 // [K][Tp][B][C]  grad wrt 1x1 conv output (for dW)
  // small per-channel gradients accumulated with atomics, [K][.]
  float *g_an_bias, *g_an_logs, *g_b_hh, *g_bf, *g_lf;
  int *flags; size_t flags_bytes;  // progress counters of the stage-pipelined kernel (nullptr: wavefront kernels only)
  // tensor-core modes, stage-pipelined kernel only: the gate / LinearZeros / 1x1-conv gradients leave the kernel as bf16
  // operand planes (same geometry as dG / dAh / dO / dzf, which may then be nullptr) and b_ih is reduced in-kernel
  void *pdG_hi, *pdG_lo, *pdAh_hi, *pdAh_lo, *pdO_hi, *pdO_lo, *pdzf_hi, *pdzf_lo;
  float *g_b_ih;
  int stash_tiled;  // st.gates / st.ahn / st.h in the tiled layout (see FwdArgs)
  // Module API (lfi_flowstep_bwd: FlowStep.forward's autograd on ONE frame): single >= 0 runs the single cell (single, t = 0)
  // with external seeds and outputs, all [B][width] for that step (the [K][Tp][B] arrays above are addressed through
  // base pointers moved back by `single` cells, the way lfi_flowstep addresses its state):
  int single;                 // -1: whole-sequence backward
  const float *dz_ext;        // [B][C]  dL/d(output of the step)          (instead of d nll / d z)
  const float *dld_ext;       // [B]     dL/d(logdet) or nullptr (0)       (instead of -dnll / ln2)
  const float *dh_ext, *dc_ext;        // [B][H] dL/d(h_out), dL/d(c_out) or nullptr (0)
  const float *h_prev_ext, *c_prev_ext;  // [B][H] state the cell started from, or nullptr (zeros)
  float *dx0_out;             // [B][C]  dL/d(input of the step)
  float *dh0_out, *dc0_out;   // [B][H]  dL/d(h_in), dL/d(c_in)
  long dg_ld; int dg_k0;      // dG row pitch / first step (0: K*GH, 0)
  // hybrid wavefronts (see FwdArgs): dh[k][t-1] += dA_h[k][t] W_hh[k] as one batched tcgen05 GEMM behind every wavefront launch;
  // the cell kernel then leaves that product out (skip_hh set by the launcher)
  WaveTc wtc;
  int skip_hh;
  // whole-sequence backward: nullptr, or [Tp][B][C] that receives dL/d(input of step 0) = dL/d(p1_face frame start_ts + t),
  // written by the cells (0, t) after their ActNorm backward (the gradient of the flow input of every frame)
  float *dx_in;
};

// The kernel that runs one direction of the flow core.
enum class CoreKernel : int {
  Wave = 0,    // anti-diagonal wavefront launches (core_fwd.cu / core_bwd.cu)
  WaveHybrid,  // the same, with the recurrent products of each wavefront as one batched tcgen05 GEMM (FwdArgs::wtc)
  Pipe,        // persistent stage pipeline, FFMA gate products (core_pipe_fwd.cu / core_pipe_bwd.cu)
  PipeTc       // persistent stage pipeline, tcgen05 gate products (core_pipe_fwd_tc.cu / core_pipe_bwd_tc.cu)
};
struct CorePlan {
  CoreKernel fwd, bwd;
  bool planes;  // the GEMM operands of the flow-step contractions are bf16 planes written by their producers (both pipelines run)
  bool tiled;   // stash (gates / ahn / h) and G in the tiled layouts of the tensor-core pipelines (fwd == PipeTc)
};
// The one place that decides the flow-core path of whole-sequence training (core_plan.cu): shape, GEMM mode, the switches of
// DESIGN.md §9.  The forward and backward calls of a training step plan alike, so they agree on the workspace layout.
CorePlan plan_core(const Dims &d, int B, int gemm_mode);
CorePlan plan_core_eval(const Dims &d, int B, int gemm_mode);  // time-chunked evaluation (lfi_seq_eval): fwd is Wave, Pipe or PipeTc

int fwd_smem_bytes(const Dims &d, int R);
int choose_rpt(const Dims &d, int B, bool bwd, bool sampler);
int choose_tile(const Dims &d, int B, bool bwd, bool sampler, int *kc_out);  // + weight-ring depth (16 or 8 rows per stage)
int launch_fwd(const FwdArgs &a, CoreKernel kern, cudaStream_t st);
int launch_inv(const InvArgs &a, cudaStream_t st);
int launch_bwd(const BwdArgs &a, CoreKernel kern, cudaStream_t st);
int launch_bwd_single(const BwdArgs &a, cudaStream_t st);  // a.single >= 0: one cell through the wavefront kernel
bool use_inv_rows(const InvArgs &a);                        // the sampler's kernel: core_inv_rows or core_inv_persistent
bool inv_rows_supported(const InvArgs &a);
int launch_inv_rows(const InvArgs &a, cudaStream_t st);

}  // namespace core
}  // namespace lfi
