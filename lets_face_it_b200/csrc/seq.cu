// Host-side orchestration of the hot path behind the C ABI (include/lfi_b200.h):
//   lfi_derive            derived weight cache
//   lfi_seq_train_fwd/bwd SeqGlow.forward (models.py:534-561) and its backward (lfi_seq_train_bwd_dx: also d input streams)
//   lfi_seq_sample        SeqGlow.inference / SeqGlow.invert (models.py:567-645)
//   lfi_flowstep          FlowStep.forward on one frame (models.py:305-373)
//   lfi_invconv_compose   InvertibleConv1x1.get_weight (modules.py:149-178) and its chain rule
// Time-parallel work (encoders, cond_transform, gate-ih, all weight gradients) goes through
// gemm_dispatch; the sequential recurrences go through the flow-core kernels.
#include "aux_kernels.cuh"
#include "core_api.cuh"
#include "core_pipe.cuh"
#include "enc_persist.cuh"
#include <algorithm>
#include <cstdlib>

namespace lfi {

size_t gemm_ws_bytes(int mode, const GemmArgs &g);  // gemm_dispatch.cu: operand-plane scratch one GEMM needs
static size_t gemm_ws_bytes_for(int mode, const GemmArgs &g) { return gemm_ws_bytes(mode, g); }
int enc_bias_grads(const float *part, int rows, int E, float *gb_ih, float *gb_hh, cudaStream_t st);  // module_grad.cu
static void *off16(void *base, size_t n) { return base ? (void *)((uint16_t *)base + n) : nullptr; }

// ------------------------------------------------------------------------------------------------
// derived cache layout (floats)
struct DerivedLayout {
  size_t Wfwd, WT, Winv, WzT, WihZ, WhhT, WfT, WcArT, WihCT, WcF, total;
};
static DerivedLayout derived_layout(const Dims &d) {
  DerivedLayout L;
  size_t o = 0;
  auto take = [&](size_t n) { size_t r = o; o += round_up_sz(n, 64); return r; };
  const size_t K = d.K;
  L.Wfwd = take(K * d.C * d.Cp);
  L.WT = take(K * d.C * d.Cp);
  L.Winv = take(K * d.C * d.Cp);
  L.WzT = take(K * d.Ci * d.GH);
  L.WihZ = take(K * d.GH * d.Cip);
  L.WhhT = take(K * d.H * d.GH);
  L.WfT = take(K * d.H * d.Cop);
  L.WcArT = take(K * d.Far * d.D);
  L.WihCT = take(K * d.D * d.GH);
  L.WcF = take(K * d.D * d.Fe);
  L.total = o;
  return L;
}

static core::DerivedView make_view(const Dims &d, const void *derived, const lfi_params *p) {
  const DerivedLayout L = derived_layout(d);
  const float *base = (const float *)derived;
  core::DerivedView v;
  v.an_bias = p->an_bias; v.an_logs = p->an_logs;
  v.Wfwd = base + L.Wfwd; v.WT = base + L.WT; v.Winv = base + L.Winv;
  v.WzT = base + L.WzT; v.WihZ = base + L.WihZ; v.WhhT = base + L.WhhT; v.Whh = p->w_hh;
  v.b_ih = p->b_ih; v.b_hh = p->b_hh; v.WfT = base + L.WfT; v.Wf = p->wf; v.bf = p->bf; v.lf = p->lf;
  v.WcArT = base + L.WcArT; v.WihCT = base + L.WihCT;
  return v;
}

// W^-1 of step k in the derived cache, [C] rows of pitch Cp (written by lfi_derive with winv); read by lfi_flowstep_rev_bwd
const float *derived_winv(const Dims &d, const void *derived, int k) {
  return (const float *)derived + derived_layout(d).Winv + (size_t)k * d.C * d.Cp;
}

static int derive_impl(const lfi_shape *s, const lfi_params *p, const float *winv, void *derived, cudaStream_t st) {
  Dims d;
  LFI_TRY(make_dims(s, &d));
  LFI_REQUIRE(p && derived, LFI_ERR_ARG, "lfi_derive: null argument");
  const DerivedLayout L = derived_layout(d);
  float *base = (float *)derived;
  const int K = d.K, C = d.C, Ci = d.Ci, GH = d.GH, H = d.H, D = d.D, Co = d.Co, In = Ci + D;
  LFI_TRY(aux::gather2d(base + L.Wfwd, d.Cp, p->w, (long)C * C, C, 1, K, C, C, st));
  LFI_TRY(aux::gather2d(base + L.WT, d.Cp, p->w, (long)C * C, 1, C, K, C, C, st));
  if (winv) LFI_TRY(aux::gather2d(base + L.Winv, d.Cp, winv, (long)C * C, C, 1, K, C, C, st));
  LFI_TRY(aux::gather2d(base + L.WzT, GH, p->w_ih, (long)GH * In, 1, In, K, Ci, GH, st));
  LFI_TRY(aux::gather2d(base + L.WihZ, d.Cip, p->w_ih, (long)GH * In, In, 1, K, GH, Ci, st));
  LFI_TRY(aux::gather2d(base + L.WhhT, GH, p->w_hh, (long)GH * H, 1, H, K, H, GH, st));
  LFI_TRY(aux::gather2d(base + L.WfT, d.Cop, p->wf, (long)Co * H, 1, H, K, H, Co, st));
  LFI_TRY(aux::gather2d(base + L.WcArT, D, p->wc, (long)D * d.F, 1, d.F, K, d.Far, D, st));
  LFI_TRY(aux::gather2d(base + L.WihCT, GH, p->w_ih + Ci, (long)GH * In, 1, In, K, D, GH, st));
  LFI_TRY(aux::fold_wc(base + L.WcF, p->wc, d, *s, st));
  return LFI_OK;
}

// ------------------------------------------------------------------------------------------------
// How the window GRU of one modality runs (plan_enc)
enum class EncStepKind {
  Unfused,  // per step: the recurrent GEMM into the shared gh scratch, then enc_gate_fwd
  Fused,    // steps s >= 1: LFI_FUSE_GRU_FWD GEMMs; step 0 (zero state): enc_gate_fwd on the xp rows
  FusedX,   // every step: a LFI_FUSE_GRU_FWD_X GEMM (input projection inside the step GEMM); step 0: the input part alone
  Persist,  // all steps in one enc_gru_fwd_persist launch (enc_persist.cu)
};
struct EncPlan {
  bool planes;       // bf16 operand planes, written by the producers themselves, never re-split
  EncStepKind step;
  bool stash;        // training: every step keeps h, gates and ahn for the backward pass (else h ping-pongs)
  bool gates16;      // the gate stash in 16-bit fixed point (the fp32 mode keeps exact fp32 gates)
};

// workspace layouts
struct EncWs {
  float *xp;     // [B*Tx][3E]
  float *hs;     // [hist][M][E]   (training) or [2][M][E] ping-pong (sampling)
  float *gates;  // [hist][M][3E]  (training only)
  float *ahn;    // [hist][M][E]   (training only)
  EncPlan plan;
  // planes only
  void *hp_hi, *hp_lo;    // h          [hist | 2][M][E]
  void *whh_hi, *whh_lo;  // W_hh       [3E][E]  (K-major B of the step GEMM, MN-major B of dh_prev = dA_h W_hh)
  // backward (training only): gate gradients of every window step, kept for the batched weight-gradient GEMMs
  float *dah32, *dan32;   // fp32 mode: [hist][M][3E], [hist][M][E]
  void *dah_hi, *dah_lo, *dan_hi, *dan_lo;  // planes, same shapes
  void *xg_hi, *xg_lo;    // masked window inputs [hist][M][round_up(dim, 8)]
  void *wih_hi, *wih_lo;  // W_ih       [3E][round_up(dim, 8)]  (input part of the fused forward step, LFI_FUSE_GRU_FWD_X)
  float *xg32;            // the same in fp32 [hist][M][dim] (split source / fp32-mode operand)
  float *dhe;             // [M][E] running d h of the window recurrence
  // Persist: xp is time-major and row-interleaved
  float *xT;              // [T*B][dim] raw frames in time-major order (input of the projection GEMM)
};

// The path of modality m's window GRU over M windows (BT raw frames), for a training call (stash for the backward pass) or not.
// The layouts (plan_enc_train, plan_sample) and every launch of build_cond, enc_bwd and seq_train_bwd follow it.
//   planes   tensor-core mode, E >= 32, E % 8 == 0, dim >= 16, M >= 128, and the step GEMM [M, E] x [E, 3E] taken by the
//            tcgen05 tiles (gemm_tc_wants): every GEMM of the encoder then runs there
//   step     Persist  not training, planes, LFI_ENC_PERSIST_SAMPLE, encp::fwd_supported, and the projection GEMM
//                     [BT, dim] x [dim, 3E] taken by the tcgen05 tiles (only those write the row-interleaved xp).  No stash to
//                     store: 4 % faster than the per-step launches
//            FusedX   training, planes, E % 64 == 0, LFI_ENC_XFUSE: the masked window inputs are gathered as operand planes in
//                     the forward pass (the backward pass needs them anyway for dW_ih) and W_ih joins the B operand
//            Fused    planes, E % 64 == 0 (the fused GRU epilogue's tile of 64 hidden units)
//            Unfused  otherwise
//   stash    training
//   gates16  training and planes
// LFI_ENC_PERSIST_SAMPLE and LFI_ENC_XFUSE are read here only, at call time.
static EncPlan plan_enc(const lfi_shape *s, int m, size_t M, size_t BT, int mode, bool training) {
  const int E = s->ehid[m], dim = s->dim[m];
  EncPlan p;
  p.planes = mode != LFI_GEMM_FP32 && E >= 32 && E % 8 == 0 && dim >= 16 && M >= 128 &&
             gemm_tc_wants(gemm_args(0, 1, (int)M, 3 * E, E, nullptr, E, nullptr, E, nullptr, 3 * E));
  const bool fused = p.planes && E % 64 == 0;
  if (!training && p.planes && env_flag("LFI_ENC_PERSIST_SAMPLE", true) && encp::fwd_supported(E, s->hist[m], M, mode) &&
      gemm_tc_wants(gemm_args(0, 1, (int)BT, 3 * E, dim, nullptr, dim, nullptr, dim, nullptr, 3 * E)))
    p.step = EncStepKind::Persist;
  else if (fused && training && env_flag("LFI_ENC_XFUSE", true))
    p.step = EncStepKind::FusedX;
  else
    p.step = fused ? EncStepKind::Fused : EncStepKind::Unfused;
  p.stash = training;
  p.gates16 = training && p.planes;
  return p;
}
static void *take_bf16(Bump &b, size_t n) { return (void *)b.take<uint16_t>(n); }
constexpr size_t kFlagInts = 1024;
struct TrainWs {
  float *cond, *Cact, *G, *ld, *gh;
  EncWs enc[LFI_NMOD];
  core::Stash st;
  // backward
  float *dx, *dh, *dc, *dG, *dAh, *dO, *dzf, *dC, *dcond, *dWcF, *xg, *dhe, *dai, *dah;
  int *flags;  // progress counters of the stage-pipelined flow core
  // flow-core kernels; with plan.planes the GEMM operands of the flow-step contractions live as bf16 planes written by their
  // producers (GEMM epilogues, core kernels), never re-split
  core::CorePlan plan;
  bool cp_lo;
  // hybrid wavefronts (plan.fwd == WaveHybrid, which a backward on hybrid wavefronts implies): W_hh planes [K][GH][H] and the
  // per-wavefront products
  void *wt_hi, *wt_lo;
  float *ghbuf;
  void *cact_hi, *cact_lo, *y_hi, *y_lo, *zf_hi, *zf_lo, *h_hi, *h_lo;
  void *dG_hi, *dG_lo, *dAh_hi, *dAh_lo, *dO_hi, *dO_lo, *dzf_hi, *dzf_lo, *dC_hi, *dC_lo;
  size_t bytes;
};

// Where the training state of a modality's encoder lives.  The training step lays all of it out in its one workspace; the module
// API (lfi_feature_encode_fwd_train / _bwd) splits it into the caller's stash (what the backward reads), forward-only scratch, the
// weight planes that each of its calls builds for itself, and backward-only scratch.  A dry-run Bump (null base) only sizes its part.
struct EncBumps { Bump *stash, *fwd, *wts, *bwd; };
static void plan_enc_train(const lfi_shape *s, int m, size_t B, size_t T, size_t M, int mode, const EncBumps &bb, EncWs &e) {
  memset(&e, 0, sizeof(EncWs));
  Bump &S = *bb.stash, &F = *bb.fwd, &W = *bb.wts, &K = *bb.bwd;
  const size_t E = s->ehid[m], h = s->hist[m];
  e.xp = F.take<float>(B * T * 3 * E);
  e.hs = S.take<float>(h * M * E);
  e.gates = S.take<float>(h * M * 3 * E);
  e.ahn = S.take<float>(h * M * E);
  e.plan = plan_enc(s, m, M, B * T, mode, true);
  if (e.plan.planes) {
    const bool lo = mode == LFI_GEMM_BF16X3;
    const size_t dimp = round_up(s->dim[m], 8);
    e.hp_hi = take_bf16(S, h * M * E);            e.hp_lo = lo ? take_bf16(S, h * M * E) : nullptr;
    e.whh_hi = take_bf16(W, 3 * E * E);           e.whh_lo = lo ? take_bf16(W, 3 * E * E) : nullptr;
    e.dah_hi = take_bf16(K, h * M * 3 * E);       e.dah_lo = lo ? take_bf16(K, h * M * 3 * E) : nullptr;
    e.dan_hi = take_bf16(K, h * M * E);           e.dan_lo = lo ? take_bf16(K, h * M * E) : nullptr;
    e.xg_hi = take_bf16(S, h * M * dimp);         e.xg_lo = lo ? take_bf16(S, h * M * dimp) : nullptr;
    e.wih_hi = take_bf16(W, 3 * E * dimp);        e.wih_lo = lo ? take_bf16(W, 3 * E * dimp) : nullptr;
  } else {
    e.dah32 = K.take<float>(h * M * 3 * E);
    e.dan32 = K.take<float>(h * M * E);
  }
  e.xg32 = K.take<float>(h * M * s->dim[m]);
  e.dhe = K.take<float>(M * E);
}

static void plan_train(const lfi_shape *s, const Dims &d, int B, int T, int mode, void *ws, TrainWs *w) {
  Bump b(ws, 0);
  const size_t Tp = T - d.start_ts, M = Tp * B, K = d.K;
  w->plan = core::plan_core(d, B, mode); w->cp_lo = mode == LFI_GEMM_BF16X3;
  const bool planes = w->plan.planes, hybrid = w->plan.fwd == core::CoreKernel::WaveHybrid;
  w->cond = b.take<float>(M * d.Fe);
  // operand-plane mode: the cond_transform activations and their gradients exist as bf16 planes only
  w->Cact = planes ? nullptr : b.take<float>(M * K * d.D);
  w->G = b.take<float>(round_up_sz(M, 32) * K * d.GH);  // (whole 32-row blocks: the row-interleaved layout of the tensor-core core)
  w->ld = b.take<float>(M);
  w->flags = b.take<int>(kFlagInts);
  size_t ghmax = 0, xgmax = 0, emax = 0;
  const EncBumps eb = {&b, &b, &b, &b};
  for (int m = 0; m < LFI_NMOD; ++m) {
    memset(&w->enc[m], 0, sizeof(EncWs));
    if (s->hist[m] <= 0 || s->ehid[m] <= 0) continue;
    const size_t E = s->ehid[m], h = s->hist[m];
    plan_enc_train(s, m, B, T, M, mode, eb, w->enc[m]);
    if (M * 3 * E > ghmax) ghmax = M * 3 * E;
    if (h * M * s->dim[m] > xgmax) xgmax = h * M * s->dim[m];
    if (E > emax) emax = E;
  }
  w->gh = b.take<float>(ghmax);
  const size_t cells = K * M;
  w->wt_hi = w->wt_lo = nullptr; w->ghbuf = nullptr;
  if (hybrid) {
    w->wt_hi = take_bf16(b, K * d.GH * d.H);
    w->wt_lo = mode == LFI_GEMM_BF16X3 ? take_bf16(b, K * d.GH * d.H) : nullptr;
    w->ghbuf = b.take<float>(2 * K * (size_t)B * d.GH);
  }
  const size_t cells_t = w->plan.tiled ? K * Tp * round_up_sz((size_t)B, 64) : cells;  // tiled stash: whole 64-sequence tiles
  w->st.y = b.take<float>(cells * d.C);
  w->st.zf = b.take<float>(cells * d.C);
  w->st.h = b.take<float>(cells_t * d.H);
  w->st.c = d.G == 4 ? b.take<float>(cells * d.H) : nullptr;
  w->st.gates = b.take<float>(cells_t * d.GH);
  w->st.ahn = d.G == 3 ? b.take<float>(cells_t * d.H) : nullptr;
  w->st.o = b.take<float>(cells * d.Co);
  w->st.xin = b.take<float>((cells + M) * d.C);
  // backward
  w->dx = b.take<float>(cells * d.C);
  w->dh = b.take<float>(cells * d.H);
  w->dc = d.G == 4 ? b.take<float>(cells * d.H) : nullptr;
  w->dG = b.take<float>(M * K * d.GH);
  w->dAh = b.take<float>(cells * d.GH);
  w->dO = b.take<float>(cells * d.Co);
  w->dzf = b.take<float>(cells * d.C);
  w->dC = planes ? nullptr : b.take<float>(M * K * d.D);
  w->dcond = b.take<float>(M * d.Fe);
  w->dWcF = b.take<float>(K * d.D * d.Fe);
  w->xg = b.take<float>(xgmax);
  w->dhe = b.take<float>(M * emax);
  w->dai = nullptr; w->dah = nullptr;
  if (planes) {
    auto two = [&](void *&hi, void *&lo_, size_t n) { hi = take_bf16(b, n); lo_ = w->cp_lo ? take_bf16(b, n) : nullptr; };
    two(w->cact_hi, w->cact_lo, M * K * d.D);
    two(w->y_hi, w->y_lo, cells * d.C); two(w->zf_hi, w->zf_lo, cells * d.C); two(w->h_hi, w->h_lo, cells * d.H);
    two(w->dG_hi, w->dG_lo, M * K * d.GH); two(w->dAh_hi, w->dAh_lo, cells * d.GH);
    two(w->dO_hi, w->dO_lo, cells * d.Co); two(w->dzf_hi, w->dzf_lo, cells * d.C);
    two(w->dC_hi, w->dC_lo, M * K * d.D);
  } else {
    w->cact_hi = w->cact_lo = w->y_hi = w->y_lo = w->zf_hi = w->zf_lo = w->h_hi = w->h_lo = nullptr;
    w->dG_hi = w->dG_lo = w->dAh_hi = w->dAh_lo = w->dO_hi = w->dO_lo = w->dzf_hi = w->dzf_lo = w->dC_hi = w->dC_lo = nullptr;
    if (hybrid) {  // hybrid wavefronts: the cells write the operands of the per-wavefront recurrent GEMMs (and of dW_hh, dWf) as planes
      const bool lo = mode == LFI_GEMM_BF16X3;
      w->h_hi = take_bf16(b, cells * d.H);      w->h_lo = lo ? take_bf16(b, cells * d.H) : nullptr;
      w->dAh_hi = take_bf16(b, cells * d.GH);   w->dAh_lo = lo ? take_bf16(b, cells * d.GH) : nullptr;
    }
  }
  w->bytes = round_up_sz(b.off, 256);
}

// Side streams / events of the fork-join sections (encoder chains, weight-gradient GEMMs).  They belong to a device: one
// lazily created set per device ordinal (a second model on another device of the same process gets its own), never destroyed
// (process lifetime, like the cached function attributes).
struct DevRes {
  bool init = false;
  cudaStream_t enc_side[LFI_NMOD] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t enc_fork = nullptr, enc_join[LFI_NMOD] = {nullptr, nullptr, nullptr, nullptr};
  cudaStream_t wg_stream = nullptr;
  cudaEvent_t wg_fork = nullptr, wg_join = nullptr, ev_dc = nullptr, ev_unfold = nullptr;
};
static int dev_res(DevRes **out) {
  constexpr int kMaxDev = 64;
  static DevRes res[kMaxDev];
  int dev = 0;
  LFI_CUDA(cudaGetDevice(&dev));
  LFI_REQUIRE(dev >= 0 && dev < kMaxDev, LFI_ERR_ARG, "device ordinal %d out of range", dev);
  DevRes &r = res[dev];
  if (!r.init) {
    for (int i = 0; i < LFI_NMOD; ++i) {
      LFI_CUDA(cudaStreamCreateWithFlags(&r.enc_side[i], cudaStreamNonBlocking));
      LFI_CUDA(cudaEventCreateWithFlags(&r.enc_join[i], cudaEventDisableTiming));
    }
    LFI_CUDA(cudaEventCreateWithFlags(&r.enc_fork, cudaEventDisableTiming));
    LFI_CUDA(cudaStreamCreateWithFlags(&r.wg_stream, cudaStreamNonBlocking));
    LFI_CUDA(cudaEventCreateWithFlags(&r.wg_fork, cudaEventDisableTiming));
    LFI_CUDA(cudaEventCreateWithFlags(&r.wg_join, cudaEventDisableTiming));
    LFI_CUDA(cudaEventCreateWithFlags(&r.ev_dc, cudaEventDisableTiming));
    LFI_CUDA(cudaEventCreateWithFlags(&r.ev_unfold, cudaEventDisableTiming));
    r.init = true;
  }
  *out = &r;
  return LFI_OK;
}
// Fork / join of n modality chains: chain i >= 1 runs on r.enc_side[i], chain 0 on st.  The join records and waits without
// checking, so that it also runs after an error.
static int enc_fork(const DevRes &r, int n, cudaStream_t st) {
  LFI_CUDA(cudaEventRecord(r.enc_fork, st));
  for (int i = 1; i < n; ++i) LFI_CUDA(cudaStreamWaitEvent(r.enc_side[i], r.enc_fork, 0));
  return LFI_OK;
}
static void enc_join(const DevRes &r, int n, cudaStream_t st) {
  for (int i = 1; i < n; ++i) {
    cudaEventRecord(r.enc_join[i], r.enc_side[i]);
    cudaStreamWaitEvent(st, r.enc_join[i], 0);
  }
}

// Encoders + "enc: none" windows into the folded feature matrix cond[M][Fe] for frames
// t = t0 .. t0+Tp-1 (ModalityEncoder / FeatureEncoder, models.py:55-80, 127-145).
//   x stream m: [B][Tx][dim] ;  skip_p1: leave the p1_face columns alone (autoregressive sampler)
//   project: also the window-independent input projections and W_hh planes (the sampler's later chunks reuse them)
//   enc[m].plan: the path of each GRU modality (plan_enc)
static int build_cond(const lfi_shape *s, const Dims &d, const lfi_params *p, const lfi_batch *bt, int t0, int Tp,
                      float *cond, EncWs *enc, float *gh, bool skip_p1, bool project, int mode, void *gws, size_t gws_bytes,
                      cudaStream_t st) {
  const int B = bt->B, T = bt->T;
  const size_t M = (size_t)Tp * B;
  const bool lo = mode == LFI_GEMM_BF16X3;
  // ---- phase 1 (caller's stream): window gathers of the "enc: none" modalities, input projections, W_hh planes ----------
  int mods[LFI_NMOD], nmods = 0;
  bool all_fused = true;
  for (int m = 0; m < LFI_NMOD; ++m) {
    const int hist = s->hist[m];
    if (hist <= 0) continue;
    if (m == 0 && skip_p1) continue;
    LFI_REQUIRE(bt->x[m], LFI_ERR_ARG, "batch: modality %d missing", m);
    const int dim = s->dim[m], E = s->ehid[m];
    if (E == 0) {
      LFI_TRY(aux::gather_windows(cond + d.enc_offe[m], d.Fe, 0, bt->x[m], bt->mask[m], B, T, dim, hist, m == 0 ? 0 : 1, t0, Tp, st));
      continue;
    }
    EncWs &ew = enc[m];
    const EncStepKind kind = ew.plan.step;
    // input projection for every raw frame (window independent): xp = x @ W_ih^T
    if (project && kind == EncStepKind::Persist) {
      // raw frames in time-major order (row tau * B + b), projected into the row-interleaved layout the persistent kernel reads
      LFI_TRY(aux::gather_windows(ew.xT, dim, 1, bt->x[m], nullptr, B, T, dim, 1, 1, 0, T, st));
      GemmArgs g = gemm_args(0, 1, B * T, 3 * E, dim, ew.xT, dim, p->enc_w_ih[m], dim, ew.xp, 3 * E);
      g.c_tiled32 = 1;
      LFI_TRY(gemm_dispatch(mode, g, gws, gws_bytes, st));
    } else if (project && kind != EncStepKind::FusedX) {  // (FusedX: inside the step GEMMs)
      GemmArgs g = gemm_args(0, 1, B * T, 3 * E, dim, bt->x[m], dim, p->enc_w_ih[m], dim, ew.xp, 3 * E);
      LFI_TRY(gemm_dispatch(mode, g, gws, gws_bytes, st));
    }
    if (ew.plan.planes && project)  // W_hh planes: once per call (weights change every optimizer step)
      LFI_TRY(split_to_planes(p->enc_w_hh[m], 3 * E, E, E, 0, 1, ew.whh_hi, lo ? ew.whh_lo : nullptr, st));
    if (kind == EncStepKind::FusedX) {
      const int dimp = round_up(dim, 8);
      LFI_TRY(aux::gather_windows_planes(ew.xg_hi, lo ? ew.xg_lo : nullptr, dimp, bt->x[m], bt->mask[m], B, T, dim, hist, 1, t0, Tp, st));
      LFI_TRY(split_to_planes(p->enc_w_ih[m], 3 * E, dim, dim, 0, 1, ew.wih_hi, lo ? ew.wih_lo : nullptr, st));
    }
    mods[nmods++] = m;
    all_fused = all_fused && kind != EncStepKind::Unfused;
  }
  // ---- phase 2: the window recurrences.  With the fused GRU launches (operands in plane form, no shared scratch) the
  //      modalities are independent chains: they run on parallel streams forked from / joined to the caller's, so that the
  //      nearly empty last wave of one launch (448 tiles on 148 persistent CTAs) is filled by the other chain's CTAs. --------
  auto chain = [&](int m, cudaStream_t cs) -> int {
    const int hist = s->hist[m], E = s->ehid[m];
    EncWs &ew = enc[m];
    const EncPlan &pl = ew.plan;
    if (pl.step == EncStepKind::Persist) {
      // persistent window GRU: all `hist` steps of a 128-window tile in one launch, state resident in shared memory
      encp::FwdArgs a;
      memset(&a, 0, sizeof(a));
      a.E = E; a.hist = hist; a.B = B; a.T = T; a.t0 = t0; a.M = (int)M; a.nplanes = lo ? 2 : 1;
      a.xp = ew.xp; a.b_ih = p->enc_b_ih[m]; a.b_hh = p->enc_b_hh[m]; a.mask = bt->mask[m];
      a.whh_hi = ew.whh_hi; a.whh_lo = lo ? ew.whh_lo : nullptr;
      a.cond = cond + d.enc_offe[m]; a.cond_ld = d.Fe;
      return encp::launch_fwd(a, cs);
    }
    for (int sidx = 0; sidx < hist; ++sidx) {
      const int cur = pl.stash ? sidx : (sidx & 1), prv = pl.stash ? sidx - 1 : ((sidx - 1) & 1);
      float *hprev = sidx ? ew.hs + (size_t)prv * M * E : nullptr, *hcur = ew.hs + (size_t)cur * M * E;
      const size_t pslot = sidx ? (size_t)prv : 0;  // (step 0 reads no state: its plane reference only shapes the tensor map)
      const PlaneRef ph = plane_ref(off16(ew.hp_hi, pslot * M * E), off16(ew.hp_lo, pslot * M * E), E);
      const PlaneRef pw = plane_ref(ew.whh_hi, ew.whh_lo, E);
      auto fill = [&](auto &q) {  // the arguments aux::EncStep and GruEpi share
        q.xp = ew.xp; q.b_ih = p->enc_b_ih[m]; q.b_hh = p->enc_b_hh[m]; q.mask = bt->mask[m]; q.hprev = hprev; q.h = hcur;
        q.gates = pl.stash ? ew.gates + (size_t)sidx * M * 3 * E : nullptr;
        q.ahn = pl.stash ? ew.ahn + (size_t)sidx * M * E : nullptr;
        q.cond = (sidx == hist - 1) ? cond + d.enc_offe[m] : nullptr; q.cond_ld = d.Fe;
        q.h_hi = off16(ew.hp_hi, (size_t)cur * M * E); q.h_lo = off16(ew.hp_lo, (size_t)cur * M * E);
        q.s = sidx; q.hist = hist; q.B = B; q.T = T; q.t0 = t0; q.E = E; q.gates16 = pl.gates16 ? 1 : 0;
      };
      auto gate_step = [&]() -> int {  // (s >= 1: after the recurrent product into the shared gh scratch)
        if (sidx) {
          GemmArgs gg = gemm_args(0, 1, (int)M, 3 * E, E, hprev, E, p->enc_w_hh[m], E, gh, 3 * E);
          if (pl.planes) { gg.pA = ph; gg.pB = pw; }
          LFI_TRY(gemm_dispatch(mode, gg, gws, gws_bytes, cs));
        }
        aux::EncStep a;
        fill(a);
        a.gh = sidx ? gh : nullptr; a.Tp = Tp;
        return aux::enc_gate_fwd(a, cs);
      };
      auto fused_step = [&](int fuse) -> int {  // recurrent product and gate math in one launch: the [M, 3E] pre-activations stay in TMEM
        GemmArgs gg = gemm_args(0, 1, (int)M, 3 * E, E, nullptr, E, nullptr, E, nullptr, 3 * E);
        gg.pA = ph; gg.pB = pw; gg.fuse = fuse;
        GruEpi &q = gg.gru;
        fill(q);
        if (fuse == LFI_FUSE_GRU_FWD_X) {
          const int dimp = round_up(s->dim[m], 8);
          q.xa_hi = off16(ew.xg_hi, (size_t)sidx * M * dimp); q.xa_lo = off16(ew.xg_lo, (size_t)sidx * M * dimp);
          q.xb_hi = ew.wih_hi; q.xb_lo = ew.wih_lo; q.xa_ld = dimp; q.xb_ld = dimp; q.xk = dimp;
          q.x_only = sidx == 0 ? 1 : 0;
        }
        return gemm_dispatch(mode, gg, gws, gws_bytes, cs);
      };
      switch (pl.step) {
        case EncStepKind::FusedX: LFI_TRY(fused_step(LFI_FUSE_GRU_FWD_X)); break;
        case EncStepKind::Fused: LFI_TRY(sidx ? fused_step(LFI_FUSE_GRU_FWD) : gate_step()); break;
        default: LFI_TRY(gate_step()); break;  // Unfused (Persist returned above)
      }
    }
    return LFI_OK;
  };
  const bool par = nmods > 1 && all_fused;
  DevRes *dr = nullptr;
  if (par) {
    LFI_TRY(dev_res(&dr));
    LFI_TRY(enc_fork(*dr, nmods, st));
  }
  int rc = LFI_OK;
  for (int i = 0; i < nmods && rc == LFI_OK; ++i) rc = chain(mods[i], par && i ? dr->enc_side[i] : st);
  if (par) enc_join(*dr, nmods, st);  // always join, also on error
  return rc;
}

// Encoder GRU of modality m, BPTT over the window (models.py:63-64), for frames t0 .. t0+Tp-1 given dcond (folded, ld Fe).  Per
// step only the gate math and dh_prev = dA_h W_hh run; the gate gradients of all steps are kept so that every weight gradient is
// ONE long-K GEMM (reduction over hist x M rows), and the bias gradients are summed inside the gate kernel.
// The training step accumulates into g (split-K GEMMs, float atomics).  o.part set (module API): the gradients are written and
// bit-reproducible - weight-gradient GEMMs with the plain store epilogue and dh_prev with ACCUM_PRE (neither ever splits K), bias
// gradients through per-block partials o.part [o.part_rows][4E] and one fixed-order reduction.  o.dx set: also dL/d(raw stream)
// [B][T][dim] through dXg = dA_h[:, :2E] W_ih[:2E] + dA_n W_ih[2E:] in o.dxg [hist*M][dim] (needs the W_ih planes in plane mode).
struct EncBwdOpts {
  float *part; int part_rows;
  float *dxg, *dx;
};
static int enc_bwd(const lfi_shape *s, const Dims &d, const lfi_params *p, const lfi_batch *bt, int t0, int Tp, int m, EncWs &ew,
                   const float *dcond, lfi_params *g, int mode, int bmode, void *gws, size_t gws_bytes, const EncBwdOpts &o,
                   cudaStream_t st) {
  const int B = bt->B, T = bt->T, hist = s->hist[m], E = s->ehid[m], dim = s->dim[m];
  const size_t M = (size_t)Tp * B;
  const bool lo = mode == LFI_GEMM_BF16X3;
  const bool det = o.part != nullptr;
  const int wepi = det ? 0 : LFI_EPI_ACCUM;
  const int dimp = round_up(dim, 8);
  if (ew.plan.step == EncStepKind::FusedX) {
    // (gathered by the forward pass, which fed them to its fused step GEMMs)
  } else if (ew.plan.planes)  // masked window inputs straight into the operand planes of the dW_ih GEMMs
    LFI_TRY(aux::gather_windows_planes(ew.xg_hi, lo ? ew.xg_lo : nullptr, dimp, bt->x[m], bt->mask[m], B, T, dim, hist, 1, t0, Tp, st));
  else
    LFI_TRY(aux::gather_windows(ew.xg32, dim, 1, bt->x[m], bt->mask[m], B, T, dim, hist, 1, t0, Tp, st));
  LFI_TRY(aux::fill(ew.dhe, 0.f, M * E, st));
  if (det) LFI_TRY(aux::fill(o.part, 0.f, (size_t)o.part_rows * 4 * E, st));
  for (int sidx = hist - 1; sidx >= 0; --sidx) {
    aux::EncStepBwd2 e;
    memset(&e, 0, sizeof(e));
    e.gates = ew.gates + (size_t)sidx * M * 3 * E; e.ahn = ew.ahn + (size_t)sidx * M * E;
    e.hprev = sidx ? ew.hs + (size_t)(sidx - 1) * M * E : nullptr;
    e.dh = ew.dhe; e.dh_extra = (sidx == hist - 1) ? dcond + d.enc_offe[m] : nullptr; e.dh_extra_ld = d.Fe;
    if (ew.plan.planes) {
      e.dah_hi = off16(ew.dah_hi, (size_t)sidx * M * 3 * E); e.dah_lo = lo ? off16(ew.dah_lo, (size_t)sidx * M * 3 * E) : nullptr;
      e.dan_hi = off16(ew.dan_hi, (size_t)sidx * M * E);     e.dan_lo = lo ? off16(ew.dan_lo, (size_t)sidx * M * E) : nullptr;
    } else {
      e.dah32 = ew.dah32 + (size_t)sidx * M * 3 * E; e.dan32 = ew.dan32 + (size_t)sidx * M * E;
    }
    e.gb_ih = g->enc_b_ih[m]; e.gb_hh = g->enc_b_hh[m]; e.M = (int)M; e.E = E; e.gates16 = ew.plan.gates16 ? 1 : 0;
    LFI_TRY(aux::enc_gate_bwd2(e, st, o.part));
    if (sidx) {  // dh_{s-1} += dA_h W_hh
      GemmArgs t = gemm_args(0, 0, (int)M, E, 3 * E, e.dah32, 3 * E, p->enc_w_hh[m], E, ew.dhe, E, det ? LFI_EPI_ACCUM_PRE : LFI_EPI_ACCUM);
      if (ew.plan.planes) { t.pA = plane_ref(e.dah_hi, e.dah_lo, 3 * E); t.pB = plane_ref(ew.whh_hi, ew.whh_lo, E); }
      LFI_TRY(gemm_dispatch(bmode, t, gws, gws_bytes, st));
    }
  }
  if (det) LFI_TRY(enc_bias_grads(o.part, o.part_rows, E, g->enc_b_ih[m], g->enc_b_hh[m], st));
  const int Kall = (int)(hist * M), Khh = (int)((hist - 1) * M);
  if (hist > 1) {  // dW_hh += sum_{s>=1} dA_h[s]^T h[s-1]
    GemmArgs q = gemm_args(1, 0, 3 * E, E, Khh, ew.dah32 ? ew.dah32 + M * 3 * E : nullptr, 3 * E, ew.hs, E, g->enc_w_hh[m], E, wepi);
    if (ew.plan.planes) { q.pA = plane_ref(off16(ew.dah_hi, M * 3 * E), lo ? off16(ew.dah_lo, M * 3 * E) : nullptr, 3 * E); q.pB = plane_ref(ew.hp_hi, ew.hp_lo, E); }
    LFI_TRY(gemm_dispatch(bmode, q, gws, gws_bytes, st));
  } else if (det) {
    LFI_CUDA(cudaMemsetAsync(g->enc_w_hh[m], 0, (size_t)3 * E * E * sizeof(float), st));
  }
  {  // dW_ih rows [0,2E) += dA_h[:, :2E]^T x  (r, u blocks coincide with the i-side gradients); rows [2E,3E) += dA_n^T x
    GemmArgs q = gemm_args(1, 0, 2 * E, dim, Kall, ew.dah32, 3 * E, ew.xg32, dim, g->enc_w_ih[m], dim, wepi);
    if (ew.plan.planes) { q.pA = plane_ref(ew.dah_hi, ew.dah_lo, 3 * E); q.pB = plane_ref(ew.xg_hi, ew.xg_lo, dimp); }
    LFI_TRY(gemm_dispatch(bmode, q, gws, gws_bytes, st));
    GemmArgs r = gemm_args(1, 0, E, dim, Kall, ew.dan32, E, ew.xg32, dim, g->enc_w_ih[m] + (size_t)2 * E * dim, dim, wepi);
    if (ew.plan.planes) { r.pA = plane_ref(ew.dan_hi, ew.dan_lo, E); r.pB = plane_ref(ew.xg_hi, ew.xg_lo, dimp); }
    LFI_TRY(gemm_dispatch(bmode, r, gws, gws_bytes, st));
  }
  if (o.dx) {  // dXg = dA_h[:, :2E] W_ih[:2E] + dA_n W_ih[2E:] (ACCUM_PRE: neither launch splits K), then the adjoint of the gather
    GemmArgs q = gemm_args(0, 0, Kall, dim, 2 * E, ew.dah32, 3 * E, p->enc_w_ih[m], dim, o.dxg, dim, 0);
    GemmArgs r = gemm_args(0, 0, Kall, dim, E, ew.dan32, E, p->enc_w_ih[m] + (size_t)2 * E * dim, dim, o.dxg, dim, LFI_EPI_ACCUM_PRE);
    if (ew.plan.planes) {
      q.pA = plane_ref(ew.dah_hi, ew.dah_lo, 3 * E); q.pB = plane_ref(ew.wih_hi, ew.wih_lo, dimp);
      r.pA = plane_ref(ew.dan_hi, ew.dan_lo, E);
      r.pB = plane_ref(off16(ew.wih_hi, (size_t)2 * E * dimp), lo ? off16(ew.wih_lo, (size_t)2 * E * dimp) : nullptr, dimp);
    }
    LFI_TRY(gemm_dispatch(bmode, q, gws, gws_bytes, st));
    LFI_TRY(gemm_dispatch(bmode, r, gws, gws_bytes, st));
    LFI_TRY(aux::window_grad(o.dx, o.dxg, dim, 1, bt->mask[m], B, T, dim, hist, 1, t0, Tp, st));
  }
  return LFI_OK;
}

// cond_transform for all K steps, then the c-part of the gate-ih product (models.py:187-190, 206-208)
static int cond_to_gates(const Dims &d, const lfi_params *p, const float *WcF, const float *cond, size_t M, float *Cact,
                         float *G, int mode, void *gws, size_t gws_bytes, cudaStream_t st, void *cact_hi = nullptr,
                         void *cact_lo = nullptr, bool g_tiled = false) {
  const int K = d.K, D = d.D, GH = d.GH, In = d.Ci + D;
  GemmArgs g = gemm_args(0, 1, (int)M, K * D, d.Fe, cond, d.Fe, WcF, d.Fe, Cact, K * D, LFI_EPI_BIAS | LFI_EPI_LRELU, p->bc);
  if (cact_hi) { g.pOut = plane_ref(cact_hi, cact_lo, K * D); g.C = nullptr; }  // the activations leave the epilogue as operand planes only
  LFI_TRY(gemm_dispatch(mode, g, gws, gws_bytes, st));
  GemmArgs h = gemm_args(0, 1, (int)M, GH, D, Cact, K * D, p->w_ih + d.Ci, In, G, K * GH, LFI_EPI_BIAS, p->b_ih);
  if (cact_hi) h.pA = plane_ref(cact_hi, cact_lo, K * D, D);
  h.batch = K; h.sA = D; h.sB = (long)GH * In; h.sC = GH; h.sBias = GH;
  if (g_tiled) { h.c_tiled32 = 1; h.sC = (long)GH * 32; }  // row-interleaved G for the tensor-core flow core (one batch = GH/4 column groups)
  LFI_TRY(gemm_dispatch(mode, h, gws, gws_bytes, st));
  return LFI_OK;
}

// Upper bound of the operand-plane scratch any single GEMM of the path needs in the tensor-core modes
// (rows = frames x sequences the time-parallel phase covers, BT = raw frames of a batch).
static size_t gemm_scratch_bound(const lfi_shape *s, const Dims &d, size_t rows, size_t BT, int mode) {
  if (mode == LFI_GEMM_FP32) return 0;
  auto mx = [](size_t a, size_t b) { return a > b ? a : b; };
  size_t emax = 0, dimmax = 0;
  for (int m = 0; m < LFI_NMOD; ++m) {
    if (s->hist[m] <= 0) continue;
    emax = mx(emax, (size_t)s->ehid[m]); dimmax = mx(dimmax, (size_t)s->dim[m]);
  }
  const size_t K = d.K, D = d.D, GH = d.GH, H = d.H, C = d.C, Co = d.Co, Fe = d.Fe;
  size_t elems = rows * K * (mx(D, GH) + mx(mx(D, H), mx(C, Co)));  // widest activation pair (dG x Cact in the dW_ih reduction)
  elems += K * D * Fe + K * GH * D + rows * Fe;                     // folded cond_transform weight, gate-ih weight, features
  elems += rows * (3 * emax + mx(emax, dimmax)) + BT * dimmax + 3 * emax * mx(emax, dimmax);  // encoders
  const size_t planes = mode == LFI_GEMM_BF16X3 ? 2 : 1;
  return round_up_sz(elems * 2 * planes + (1 << 16), 256);
}

static int check_batch(const lfi_shape *s, const Dims &d, const lfi_batch *b, int min_T) {
  LFI_REQUIRE(b && b->B >= 1, LFI_ERR_ARG, "batch: B must be >= 1");
  LFI_REQUIRE(b->T >= min_T, LFI_ERR_SHAPE, "batch: T=%d shorter than needed (%d)", b->T, min_T);
  (void)s; (void)d;
  return LFI_OK;
}

}  // namespace lfi

using namespace lfi;

static cudaEvent_t g_grad_ready_event = nullptr;

extern "C" {

int lfi_set_grad_ready_event(void *event) { g_grad_ready_event = (cudaEvent_t)event; return LFI_OK; }
static cudaEvent_t g_derived_ready_event = nullptr;
int lfi_set_derived_ready_event(void *event) { g_derived_ready_event = (cudaEvent_t)event; return LFI_OK; }

int lfi_feature_dim(const lfi_shape *s) { Dims d; return make_dims(s, &d) == LFI_OK ? d.F : -1; }
int lfi_feature_dim_folded(const lfi_shape *s) { Dims d; return make_dims(s, &d) == LFI_OK ? d.Fe : -1; }
int lfi_start_ts(const lfi_shape *s) { Dims d; return make_dims(s, &d) == LFI_OK ? d.start_ts : -1; }
int lfi_coupling_out(const lfi_shape *s) { Dims d; return make_dims(s, &d) == LFI_OK ? d.Co : -1; }

size_t lfi_derived_bytes(const lfi_shape *s) {
  Dims d;
  if (make_dims(s, &d) != LFI_OK) return 0;
  return derived_layout(d).total * sizeof(float);
}

int lfi_derive(const lfi_shape *s, const lfi_params *p, const float *winv, void *derived, int gemm_mode, void *stream) {
  (void)gemm_mode;
  return derive_impl(s, p, winv, derived, (cudaStream_t)stream);
}

size_t lfi_train_ws_bytes(const lfi_shape *s, int B, int T, int gemm_mode) {
  Dims d;
  if (make_dims(s, &d) != LFI_OK || T <= d.start_ts || B < 1) return 0;
  TrainWs w;
  plan_train(s, d, B, T, gemm_mode, nullptr, &w);
  return w.bytes + gemm_scratch_bound(s, d, (size_t)(T - d.start_ts) * B, (size_t)B * T, gemm_mode);
}

int lfi_seq_train_fwd(const lfi_shape *s, const void *derived, const lfi_params *p, const lfi_batch *bt, float *z,
                      float *nll, float *scale_out, void *ws, size_t ws_bytes, int gemm_mode, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  Dims d;
  LFI_TRY(make_dims(s, &d));
  LFI_REQUIRE(derived && p && z && nll && ws, LFI_ERR_ARG, "lfi_seq_train_fwd: null argument");
  LFI_TRY(check_batch(s, d, bt, d.start_ts + 1));
  const int B = bt->B, T = bt->T, Tp = T - d.start_ts;
  const size_t M = (size_t)Tp * B;
  TrainWs w;
  plan_train(s, d, B, T, gemm_mode, ws, &w);
  const size_t gneed = gemm_scratch_bound(s, d, M, (size_t)B * T, gemm_mode);
  LFI_REQUIRE(ws_bytes >= w.bytes + gneed, LFI_ERR_WORKSPACE, "train workspace too small: %zu < %zu", ws_bytes, w.bytes + gneed);
  void *gws = (char *)ws + w.bytes;
  const size_t gws_bytes = ws_bytes - w.bytes;
  const DerivedLayout L = derived_layout(d);
  const float *WcF = (const float *)derived + L.WcF;

  LFI_TRY(build_cond(s, d, p, bt, d.start_ts, Tp, w.cond, w.enc, w.gh, false, true, gemm_mode, gws, gws_bytes, st));
  // the encoders read their parameters directly; the derived cache (composed 1x1 weights, folded W_c, transposes) is first needed
  // here - a caller that rebuilds it on another stream hands over the event to wait for (lfi_set_derived_ready_event)
  if (g_derived_ready_event) LFI_CUDA(cudaStreamWaitEvent(st, g_derived_ready_event, 0));
  LFI_TRY(cond_to_gates(d, p, WcF, w.cond, M, w.Cact, w.G, gemm_mode, gws, gws_bytes, st, w.plan.planes ? w.cact_hi : nullptr,
                        w.plan.planes ? w.cact_lo : nullptr, w.plan.tiled));

  core::FwdArgs a;
  memset(&a, 0, sizeof(a));
  a.d = d; a.dv = make_view(d, derived, p); a.B = B; a.Tp = Tp; a.k_first = 0; a.k_last = d.K - 1;
  a.x0 = bt->x[0] + (size_t)d.start_ts * d.C; a.x_sb = (long)T * d.C; a.x_st = d.C;
  a.G = w.G; a.g_ld = (long)d.K * d.GH; a.g_k0 = 0;
  a.xin = w.st.xin; a.st_y = w.st.y; a.st_zf = w.st.zf; a.st_h = w.st.h; a.st_c = w.st.c; a.st_gates = w.st.gates;
  a.st_ahn = w.st.ahn; a.st_o = w.st.o; a.ld = w.ld; a.ld_accumulate = 0; a.nll = nll; a.z_out = z;
  a.scale_out = scale_out;
  a.flags = w.flags; a.flags_bytes = kFlagInts * sizeof(int);
  if (w.plan.planes) { a.py_hi = w.y_hi; a.py_lo = w.y_lo; a.pzf_hi = w.zf_hi; a.pzf_lo = w.zf_lo; a.ph_hi = w.h_hi; a.ph_lo = w.h_lo; }
  a.stash_tiled = w.plan.tiled ? 1 : 0;
  a.g_tiled = w.plan.tiled ? 1 : 0;
  if (w.plan.fwd == core::CoreKernel::WaveHybrid) {  // recurrent weights as operand planes, once per call (they change with every optimizer step)
    a.ph_hi = w.h_hi; a.ph_lo = w.h_lo;
    LFI_TRY(split_to_planes(p->w_hh, d.GH, d.H, d.H, (long)d.GH * d.H, d.K, w.wt_hi, w.wt_lo, st));
    a.wtc.mode = gemm_mode; a.wtc.whh_hi = w.wt_hi; a.wtc.whh_lo = w.wt_lo; a.wtc.ghbuf = w.ghbuf; a.wtc.gws = gws; a.wtc.gws_bytes = gws_bytes;
  }
  return core::launch_fwd(a, w.plan.fwd, st);
}

// Backward of lfi_seq_train_fwd.  dx == nullptr: parameter gradients only (lfi_seq_train_bwd).  Otherwise (lfi_seq_train_bwd_dx)
// also dL/d(raw stream m) into every non-null dx[m] [B][T][dim]: the flow core keeps the gradient of its input (step 0), d cond is
// formed for the "enc: none" columns as well, and the window adjoints (aux::window_grad, inside enc_bwd for the GRU modalities)
// scatter d cond back onto the frames; dws holds the dXg scratch of each GRU modality (plan_train_dx).
struct TrainDxWs { float *dxg[LFI_NMOD]; size_t bytes; };
static void plan_train_dx(const lfi_shape *s, size_t M, void *dws, TrainDxWs *x) {
  Bump b(dws, 0);
  for (int m = 0; m < LFI_NMOD; ++m)
    x->dxg[m] = (s->hist[m] > 0 && s->ehid[m] > 0) ? b.take<float>((size_t)s->hist[m] * M * s->dim[m]) : nullptr;
  x->bytes = round_up_sz(b.off > 256 ? b.off : 256, 256);
}

static int seq_train_bwd(const lfi_shape *s, const void *derived, const lfi_params *p, const lfi_batch *bt, const float *z,
                         const float *dnll, lfi_params *g, void *ws, size_t ws_bytes, int gemm_mode, cudaStream_t st,
                         float *const *dx, void *dws, size_t dws_bytes, const char *what) {
  Dims d;
  LFI_TRY(make_dims(s, &d));
  LFI_REQUIRE(derived && p && z && dnll && g && ws, LFI_ERR_ARG, "%s: null argument", what);
  LFI_TRY(check_batch(s, d, bt, d.start_ts + 1));
  const int B = bt->B, T = bt->T, Tp = T - d.start_ts, K = d.K, C = d.C, Ci = d.Ci, GH = d.GH, H = d.H, D = d.D, Co = d.Co;
  const int In = Ci + D;
  const size_t M = (size_t)Tp * B;
  TrainWs w;
  plan_train(s, d, B, T, gemm_mode, ws, &w);
  LFI_REQUIRE(ws_bytes >= w.bytes + gemm_scratch_bound(s, d, M, (size_t)B * T, gemm_mode), LFI_ERR_WORKSPACE, "train workspace too small");
  TrainDxWs xw;
  memset(&xw, 0, sizeof(xw));
  bool none_dx = false;  // an "enc: none" modality wants the gradient of its stream
  if (dx) {
    for (int m = 0; m < LFI_NMOD; ++m) {
      LFI_REQUIRE(!dx[m] || s->hist[m] > 0, LFI_ERR_ARG, "%s: dx[%d] given for an absent modality", what, m);
      none_dx = none_dx || (dx[m] && s->ehid[m] == 0);
    }
    plan_train_dx(s, M, dws, &xw);
    LFI_REQUIRE(dws, LFI_ERR_ARG, "%s: null dx workspace", what);
    LFI_REQUIRE(dws_bytes >= xw.bytes, LFI_ERR_WORKSPACE, "%s: dx workspace too small: %zu < %zu", what, dws_bytes, xw.bytes);
  }
  void *gws = (char *)ws + w.bytes;
  const size_t gws_bytes = ws_bytes - w.bytes;
  const DerivedLayout L = derived_layout(d);
  const float *WcF = (const float *)derived + L.WcF;

  // Numerics of the time-parallel backward GEMMs: the mode of the call, or (LFI_BWD_BF16=1, an option measured next to the
  // parity mode, not its default) single bf16 products on the hi planes while the forward pass and the flow core keep split-bf16
  const int bmode = (gemm_mode == LFI_GEMM_BF16X3 && env_flag("LFI_BWD_BF16", false)) ? LFI_GEMM_BF16 : gemm_mode;
  // 1. sequential core, reverse wavefronts
  core::BwdArgs a;
  memset(&a, 0, sizeof(a));
  a.single = -1;
  a.d = d; a.dv = make_view(d, derived, p); a.B = B; a.Tp = Tp; a.dnll = dnll; a.z = z; a.st = w.st;
  a.dx = w.dx; a.dh = w.dh; a.dc = w.dc; a.dG = w.dG; a.dAh = w.dAh; a.dO = w.dO; a.dzf = w.dzf;
  a.g_an_bias = g->an_bias; a.g_an_logs = g->an_logs; a.g_b_hh = g->b_hh; a.g_bf = g->bf; a.g_lf = g->lf;
  a.flags = w.flags; a.flags_bytes = kFlagInts * sizeof(int);
  const bool hybrid = w.plan.fwd == core::CoreKernel::WaveHybrid;
  if (w.plan.planes) {
    a.dG = nullptr; a.dAh = nullptr; a.dO = nullptr; a.dzf = nullptr;
    a.pdG_hi = w.dG_hi; a.pdG_lo = w.dG_lo; a.pdAh_hi = w.dAh_hi; a.pdAh_lo = w.dAh_lo;
    a.pdO_hi = w.dO_hi; a.pdO_lo = w.dO_lo; a.pdzf_hi = w.dzf_hi; a.pdzf_lo = w.dzf_lo;
    a.g_b_ih = g->b_ih;
  }
  a.stash_tiled = w.plan.tiled ? 1 : 0;
  if (hybrid) {  // the cells write dA_h as operand planes only; the planes of W_hh were built by the forward call of this step
    a.pdAh_hi = w.dAh_hi; a.pdAh_lo = w.dAh_lo; a.dAh = nullptr;
    a.wtc.mode = gemm_mode; a.wtc.whh_hi = w.wt_hi; a.wtc.whh_lo = w.wt_lo; a.wtc.ghbuf = w.ghbuf; a.wtc.gws = gws; a.wtc.gws_bytes = gws_bytes;
  }
  // d(flow input) of every frame into the step-0 slot of the hand-off buffer, which nothing else writes or reads
  float *dflow = (dx && dx[0]) ? w.dx : nullptr;
  a.dx_in = dflow;
  LFI_TRY(core::launch_bwd(a, w.plan.bwd, st));

  // 2. weight gradients of the per-step matrices as batched (over k) reductions over the M rows.  With every operand in
  //    plane form (no shared scratch) they are independent of the rest of the backward pass: they run on a side stream,
  //    concurrently with the cond_transform / encoder backward below (small-output long-K launches and a latency-bound
  //    chain fill each other's idle SMs), and are joined before the call returns.
  DevRes *dr = nullptr;
  LFI_TRY(dev_res(&dr));
  cudaStream_t wg_stream = dr->wg_stream;
  cudaEvent_t wg_fork = dr->wg_fork, wg_join = dr->wg_join;
  const bool wg_par = w.plan.planes;
  cudaStream_t st_main = st;
  if (wg_par) {
    LFI_CUDA(cudaEventRecord(wg_fork, st_main));
    LFI_CUDA(cudaStreamWaitEvent(wg_stream, wg_fork, 0));
    st = wg_stream;
  }
  auto join_wgrads = [&]() {
    if (wg_par) { cudaEventRecord(wg_join, wg_stream); cudaStreamWaitEvent(st_main, wg_join, 0); }
  };
  auto wgrad = [&](int Mo, int No, size_t red, const float *A, int lda, long sA, const float *Bm, int ldb, long sB, float *Cm,
                   int ldc, long sC, PlaneRef pa = PlaneRef{nullptr, nullptr, 0, 0}, PlaneRef pb = PlaneRef{nullptr, nullptr, 0, 0}) -> int {
    GemmArgs q = gemm_args(1, 0, Mo, No, (int)red, A, lda, Bm, ldb, Cm, ldc, LFI_EPI_ACCUM);
    q.batch = K; q.sA = sA; q.sB = sB; q.sC = sC;
    if (w.plan.planes || hybrid) { q.pA = pa; q.pB = pb; }  // (a plane reference with a null pointer means: split the fp32 operand)
    return gemm_dispatch(bmode, q, gws, gws_bytes, st);
  };
  const PlaneRef pdG = plane_ref(w.dG_hi, w.dG_lo, K * GH, GH), ph = plane_ref(w.h_hi, w.h_lo, H, (long)(M * H));
  if (Tp > 1)  // dW_hh[k] += dA_h[k][t>=1]^T h[k][t-1]
    LFI_TRY(wgrad(GH, H, (size_t)(Tp - 1) * B, w.dAh + (size_t)B * GH, GH, (long)(M * GH), w.st.h, H, (long)(M * H), g->w_hh, H,
                  (long)GH * H, plane_ref(off16(w.dAh_hi, (size_t)B * GH), off16(w.dAh_lo, (size_t)B * GH), GH, (long)(M * GH)), ph));
  LFI_TRY(wgrad(GH, Ci, M, w.dG, K * GH, GH, w.st.zf, C, (long)(M * C), g->w_ih, In, (long)GH * In, pdG,
                plane_ref(w.zf_hi, w.zf_lo, C, (long)(M * C))));                                                      // dW_ih[:, :Ci]
  LFI_TRY(wgrad(GH, D, M, w.dG, K * GH, GH, w.Cact, K * D, D, g->w_ih + Ci, In, (long)GH * In, pdG,
                plane_ref(w.cact_hi, w.cact_lo, K * D, D)));                                                          // dW_ih[:, Ci:]
  LFI_TRY(wgrad(Co, H, M, w.dO, Co, (long)(M * Co), w.st.h, H, (long)(M * H), g->wf, H, (long)Co * H,
                plane_ref(w.dO_hi, w.dO_lo, Co, (long)(M * Co)), ph));                                                 // dWf
  LFI_TRY(wgrad(C, C, M, w.st.y, C, (long)(M * C), w.dzf, C, (long)(M * C), g->w, C, (long)C * C,
                plane_ref(w.y_hi, w.y_lo, C, (long)(M * C)), plane_ref(w.dzf_hi, w.dzf_lo, C, (long)(M * C))));       // dW (1x1 conv)
  if (!w.plan.planes) LFI_TRY(aux::colsum(g->b_ih, w.dG, K * GH, (int)M, K * GH, 1.0f, st));  // (planes: reduced inside the core kernel ...
  if (w.plan.bwd == core::CoreKernel::PipeTc) {
    // ... except with the tensor-core backward pipeline, which leaves the RNN bias gradients to column sums of its planes:
    // d b_ih = colsum(dG) (r, u parts also are d b_hh's), d b_hh n part = colsum of the n columns of dA_h)
    LFI_TRY(aux::colsum_planes(g->b_ih, g->b_hh, GH, 2 * H, 0, w.dG_hi, w.cp_lo ? w.dG_lo : nullptr, K * GH, 0, 1, (int)M, 0, K * GH, st));
    LFI_TRY(aux::colsum_planes(g->b_hh + 2 * H, nullptr, 1, 0, GH, w.dAh_hi, w.cp_lo ? w.dAh_lo : nullptr, GH, (long)(M * GH), K, (int)M, 2 * H, H, st));
  }
  st = st_main;

  // 3. cond_transform backward
  {
    GemmArgs q = gemm_args(0, 0, (int)M, D, GH, w.dG, K * GH, p->w_ih + Ci, In, w.dC, K * D, LFI_EPI_LRELU_BWD);
    q.batch = K; q.sA = GH; q.sB = (long)GH * In; q.sC = D; q.aux = w.Cact; q.ldaux = K * D; q.sAux = D;
    if (w.plan.planes) {  // planes in, planes out; LeakyReLU' from the sign of the activation plane; d b_c reduced in the epilogue
      q.pA = pdG; q.pOut = plane_ref(w.dC_hi, w.dC_lo, K * D, D); q.C = nullptr;
      q.aux = nullptr; q.auxp = w.cact_hi; q.ldauxp = K * D; q.sAuxp = D;
      q.colsum = g->bc; q.sColsum = D;
    }
    LFI_TRY(gemm_dispatch(bmode, q, gws, gws_bytes, st));
    if (!w.plan.planes) LFI_TRY(aux::colsum(g->bc, w.dC, K * D, (int)M, K * D, 1.0f, st));
    // d W_c = dC^T cond: not needed by the rest of the backward pass.  With the side stream available it runs there, next to the
    // encoder backward (its operand-plane scratch sits behind the region the d cond GEMM of the main stream uses).
    GemmArgs r = gemm_args(1, 0, K * D, d.Fe, (int)M, w.dC, K * D, w.cond, d.Fe, w.dWcF, d.Fe, 0);
    if (w.plan.planes) r.pA = plane_ref(w.dC_hi, w.dC_lo, K * D);
    size_t side_off = 0;
    bool wc_side = false;
    if (wg_par) {
      GemmArgs qd = gemm_args(0, 0, (int)M, d.Fe, K * D, nullptr, K * D, WcF, d.Fe, nullptr, d.Fe, 0);
      side_off = round_up_sz(gemm_ws_bytes_for(gemm_mode, qd), 1024);
      wc_side = side_off + gemm_ws_bytes_for(gemm_mode, r) <= gws_bytes;
    }
    if (wc_side) {
      cudaEvent_t ev_dc = dr->ev_dc;
      LFI_CUDA(cudaEventRecord(ev_dc, st));
      LFI_CUDA(cudaStreamWaitEvent(wg_stream, ev_dc, 0));
      LFI_TRY(gemm_dispatch(bmode, r, (char *)gws + side_off, gws_bytes - side_off, wg_stream));
      LFI_TRY(aux::unfold_wc_grad(g->wc, w.dWcF, d, *s, wg_stream));
      if (g_grad_ready_event) LFI_CUDA(cudaEventRecord(g_grad_ready_event, wg_stream));  // every flow-step weight gradient is final
    } else {
      LFI_TRY(gemm_dispatch(bmode, r, gws, gws_bytes, st));
      LFI_TRY(aux::unfold_wc_grad(g->wc, w.dWcF, d, *s, st));
      if (g_grad_ready_event) {  // data parallel: every flow-step weight gradient is final here, once the side-stream GEMMs are too
        if (wg_par) {  // record on the side stream, ordered after this point of the main stream (no early join of the main stream)
          cudaEvent_t ev_unfold = dr->ev_unfold;
          LFI_CUDA(cudaEventRecord(ev_unfold, st));
          LFI_CUDA(cudaStreamWaitEvent(wg_stream, ev_unfold, 0));
          LFI_CUDA(cudaEventRecord(g_grad_ready_event, wg_stream));
        } else {
          LFI_CUDA(cudaEventRecord(g_grad_ready_event, st));
        }
      }
    }
  }
  // d cond for the encoder columns [enc_lo, Fe)
  int enc_lo = -1;
  for (int m = 0; m < LFI_NMOD; ++m)
    if (s->hist[m] > 0 && s->ehid[m] > 0) { enc_lo = d.enc_offe[m]; break; }
  if (enc_lo < 0 && !none_dx) { join_wgrads(); return LFI_OK; }
  auto dcond_gemm = [&](int lo, int hi) -> int {
    GemmArgs q = gemm_args(0, 0, (int)M, hi - lo, K * D, w.dC, K * D, WcF + lo, d.Fe, w.dcond + lo, d.Fe, 0);
    if (w.plan.planes) q.pA = plane_ref(w.dC_hi, w.dC_lo, K * D);
    return gemm_dispatch(bmode, q, gws, gws_bytes, st);
  };
  if (enc_lo >= 0) LFI_TRY(dcond_gemm(enc_lo, d.Fe));
  // "enc: none" streams: d cond of the columns before enc_lo in a launch of its own (one GEMM over all Fe columns would change the
  // tile split, and in the tensor-core modes the numerics, of the encoder columns), then the adjoint of the window gather (p1_face:
  // its window excludes frame t, and the gradient of the flow input of frame start_ts + t' joins the same fixed-order sum).
  // Reads only final values: dC and the flow-core output.
  auto none_grads = [&]() -> int {
    if (none_dx && enc_lo != 0) LFI_TRY(dcond_gemm(0, enc_lo < 0 ? d.Fe : enc_lo));
    for (int m = 0; dx && m < LFI_NMOD; ++m)
      if (dx[m] && s->ehid[m] == 0)
        LFI_TRY(aux::window_grad(dx[m], w.dcond + d.enc_offe[m], d.Fe, 0, bt->mask[m], B, T, s->dim[m], s->hist[m], m == 0 ? 0 : 1,
                                 d.start_ts, Tp, st, m == 0 ? dflow : nullptr));
    return LFI_OK;
  };

  // 4. encoder GRUs, BPTT over the window (enc_bwd).  The modalities are independent chains of a latency-bound GEMM and an
  //    HBM-bound gate kernel per window step: with every operand in plane form (no shared scratch) they run on parallel streams
  //    forked from / joined to the caller's.
  //    With dx[m] set the chain also forms dL/d(stream m) (EncBwdOpts.dx, its own dXg scratch: the chains run concurrently).
  auto enc_chain = [&](int m, cudaStream_t cs) -> int {
    float *dxm = dx ? dx[m] : nullptr;
    EncWs &ew = w.enc[m];
    if (dxm && ew.plan.planes && ew.plan.step != EncStepKind::FusedX)  // (FusedX: the forward steps built the W_ih planes)
      LFI_TRY(split_to_planes(p->enc_w_ih[m], 3 * s->ehid[m], s->dim[m], s->dim[m], 0, 1, ew.wih_hi,
                              gemm_mode == LFI_GEMM_BF16X3 ? ew.wih_lo : nullptr, cs));
    const EncBwdOpts o = {nullptr, 0, dxm ? xw.dxg[m] : nullptr, dxm};
    return enc_bwd(s, d, p, bt, d.start_ts, Tp, m, ew, w.dcond, g, gemm_mode, bmode, gws, gws_bytes, o, cs);
  };
  int mods[LFI_NMOD], nmods = 0;
  bool all_planes = true;
  for (int m = 0; m < LFI_NMOD; ++m)
    if (s->hist[m] > 0 && s->ehid[m] > 0) { mods[nmods++] = m; all_planes = all_planes && w.enc[m].plan.planes; }
  const bool par = nmods > 1 && all_planes;
  if (par) LFI_TRY(enc_fork(*dr, nmods, st));
  int rc = LFI_OK;
  for (int i = 0; i < nmods && rc == LFI_OK; ++i) rc = enc_chain(mods[i], par && i ? dr->enc_side[i] : st);
  if (rc == LFI_OK) rc = none_grads();
  if (par) enc_join(*dr, nmods, st);  // always join, also on error
  join_wgrads();
  return rc;
}

int lfi_seq_train_bwd(const lfi_shape *s, const void *derived, const lfi_params *p, const lfi_batch *bt, const float *z,
                      const float *dnll, lfi_params *g, void *ws, size_t ws_bytes, int gemm_mode, void *stream) {
  return seq_train_bwd(s, derived, p, bt, z, dnll, g, ws, ws_bytes, gemm_mode, (cudaStream_t)stream, nullptr, nullptr, 0,
                       "lfi_seq_train_bwd");
}

size_t lfi_train_dx_ws_bytes(const lfi_shape *s, int B, int T, int gemm_mode) {
  (void)gemm_mode;  // (the dXg scratch is fp32 in every mode)
  Dims d;
  if (make_dims(s, &d) != LFI_OK || T <= d.start_ts || B < 1) return 0;
  TrainDxWs x;
  plan_train_dx(s, (size_t)(T - d.start_ts) * B, nullptr, &x);
  return x.bytes;
}

int lfi_seq_train_bwd_dx(const lfi_shape *s, const void *derived, const lfi_params *p, const lfi_batch *bt, const float *z,
                         const float *dnll, lfi_params *g, void *ws, size_t ws_bytes, float *const dx[LFI_NMOD], void *dws,
                         size_t dws_bytes, int gemm_mode, void *stream) {
  LFI_REQUIRE(dx, LFI_ERR_ARG, "lfi_seq_train_bwd_dx: null dx");
  return seq_train_bwd(s, derived, p, bt, z, dnll, g, ws, ws_bytes, gemm_mode, (cudaStream_t)stream, dx, dws, dws_bytes,
                       "lfi_seq_train_bwd_dx");
}

// ------------------------------------------------------------------------------------------------
// sampling / invert
struct SampleWs {
  float *cond, *Cs, *G, *gh, *hstate, *cstate;
  EncWs enc[LFI_NMOD];
  // tensor-core modes, autoregressive sampling: per-frame conditioning GEMMs (see lfi_seq_sample)
  bool tc_ar;
  float *car;                       // [B][Far]   p1_face window of the current frame
  void *war_hi, *war_lo;            // [K*D][Far] autoregressive columns of the folded cond_transform weight
  void *wihc_hi, *wihc_lo;          // [K][GH][D] W_ih[:, Ci:]
  void *cact_hi, *cact_lo;          // [B][K*D]   cond_transform activations of the current frame
  size_t bytes;
};
static bool sample_tc_ar(const Dims &d, int mode) {
  return mode != LFI_GEMM_FP32 && d.Far > 0 && d.Far % 8 == 0 && d.D % 8 == 0;
}
// The encoders of a call without gradients over chunks of Mc windows (sampling, feature encoding, evaluation): the input
// projections of all B*T raw frames (computed once per call), the window state ping-pong, and the shared gh scratch.
static void plan_enc_nograd(const lfi_shape *s, int B, int T, size_t Mc, int mode, Bump &b, EncWs *enc, float **gh) {
  size_t ghmax = 0;
  for (int m = 0; m < LFI_NMOD; ++m) {
    memset(&enc[m], 0, sizeof(EncWs));
    if (s->hist[m] <= 0 || s->ehid[m] <= 0) continue;
    const size_t E = s->ehid[m];
    EncWs &e = enc[m];
    e.xp = b.take<float>(encp::tiled_rows((size_t)B * T) * 3 * E);
    e.hs = b.take<float>(2 * Mc * E);
    e.plan = plan_enc(s, m, Mc, (size_t)B * T, mode, false);
    e.xT = e.plan.step == EncStepKind::Persist ? b.take<float>((size_t)B * T * s->dim[m]) : nullptr;
    if (e.plan.planes) {
      const bool lo = mode == LFI_GEMM_BF16X3;
      e.hp_hi = take_bf16(b, 2 * Mc * E);  e.hp_lo = lo ? take_bf16(b, 2 * Mc * E) : nullptr;
      e.whh_hi = take_bf16(b, 3 * E * E);  e.whh_lo = lo ? take_bf16(b, 3 * E * E) : nullptr;
    }
    if (Mc * 3 * E > ghmax) ghmax = Mc * 3 * E;
  }
  *gh = b.take<float>(ghmax);
}
static void plan_sample(const lfi_shape *s, const Dims &d, int B, int T, int chunk, int mode, void *ws, SampleWs *w) {
  Bump b(ws, 0);
  const size_t Mc = (size_t)chunk * B, K = d.K;
  w->cond = b.take<float>(Mc * d.Fe);
  w->Cs = b.take<float>(Mc * K * d.D);
  w->G = b.take<float>(Mc * K * d.GH);
  w->hstate = b.take<float>(K * B * d.H);
  w->cstate = d.G == 4 ? b.take<float>(K * B * d.H) : nullptr;
  plan_enc_nograd(s, B, T, Mc, mode, b, w->enc, &w->gh);
  w->tc_ar = sample_tc_ar(d, mode);
  if (w->tc_ar) {
    const bool lo = mode == LFI_GEMM_BF16X3;
    w->car = b.take<float>((size_t)B * d.Far);
    w->war_hi = take_bf16(b, K * d.D * d.Far);            w->war_lo = lo ? take_bf16(b, K * d.D * d.Far) : nullptr;
    w->wihc_hi = take_bf16(b, K * d.GH * d.D);            w->wihc_lo = lo ? take_bf16(b, K * d.GH * d.D) : nullptr;
    w->cact_hi = take_bf16(b, (size_t)B * K * d.D);       w->cact_lo = lo ? take_bf16(b, (size_t)B * K * d.D) : nullptr;
  }
  w->bytes = round_up_sz(b.off, 256);
}

// FeatureEncoder.forward (models.py:127-145) for frames t0 .. t0+Tp-1 of a batch: folded features [Tp*B][Fe]
size_t lfi_feature_ws_bytes(const lfi_shape *s, int B, int T, int Tp, int gemm_mode) {
  Dims d;
  if (make_dims(s, &d) != LFI_OK || B < 1 || Tp < 1) return 0;
  SampleWs w;
  plan_sample(s, d, B, T, Tp, gemm_mode, nullptr, &w);
  return w.bytes + gemm_scratch_bound(s, d, (size_t)Tp * B, (size_t)B * T, gemm_mode);
}

int lfi_feature_encode(const lfi_shape *s, const lfi_params *p, const lfi_batch *bt, int t0, int Tp, float *cond, void *ws,
                       size_t ws_bytes, int gemm_mode, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  Dims d;
  LFI_TRY(make_dims(s, &d));
  LFI_REQUIRE(p && bt && cond && ws, LFI_ERR_ARG, "lfi_feature_encode: null argument");
  LFI_REQUIRE(t0 >= d.start_ts && t0 + Tp <= bt->T && Tp >= 1, LFI_ERR_SHAPE, "lfi_feature_encode: frames [%d,%d) outside [%d,%d)", t0,
              t0 + Tp, d.start_ts, bt->T);
  SampleWs w;
  plan_sample(s, d, bt->B, bt->T, Tp, gemm_mode, ws, &w);
  LFI_REQUIRE(ws_bytes >= w.bytes + gemm_scratch_bound(s, d, (size_t)Tp * bt->B, (size_t)bt->B * bt->T, gemm_mode), LFI_ERR_WORKSPACE,
              "feature workspace too small");
  void *gws = (char *)ws + w.bytes;
  return build_cond(s, d, p, bt, t0, Tp, cond, w.enc, w.gh, false, true, gemm_mode, gws, ws_bytes - w.bytes, st);
}

size_t lfi_sample_ws_bytes(const lfi_shape *s, int B, int T, int chunk, int gemm_mode) {
  Dims d;
  if (make_dims(s, &d) != LFI_OK || B < 1 || chunk < 1) return 0;
  SampleWs w;
  plan_sample(s, d, B, T, chunk, gemm_mode, nullptr, &w);
  return w.bytes + gemm_scratch_bound(s, d, (size_t)chunk * B, (size_t)B * T, gemm_mode);
}

int lfi_seq_sample(const lfi_shape *s, const void *derived, const lfi_params *p, const lfi_batch *bt, int seq_len,
                   const float *noise, float *faces, float *logdet_out, int teacher_forced, int chunk, void *ws,
                   size_t ws_bytes, int gemm_mode, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  Dims d;
  LFI_TRY(make_dims(s, &d));
  LFI_REQUIRE(derived && p && faces && ws && chunk >= 1, LFI_ERR_ARG, "lfi_seq_sample: null argument");
  LFI_TRY(check_batch(s, d, bt, seq_len));
  LFI_REQUIRE(seq_len > d.start_ts, LFI_ERR_SHAPE, "seq_len=%d must exceed the longest history %d", seq_len, d.start_ts);
  const int B = bt->B, T = bt->T, Tgen = seq_len - d.start_ts, K = d.K;
  SampleWs w;
  plan_sample(s, d, B, T, chunk, gemm_mode, ws, &w);
  const size_t gneed = gemm_scratch_bound(s, d, (size_t)chunk * B, (size_t)B * T, gemm_mode);
  LFI_REQUIRE(ws_bytes >= w.bytes + gneed, LFI_ERR_WORKSPACE, "sample workspace too small: %zu < %zu", ws_bytes, w.bytes + gneed);
  void *gws = (char *)ws + w.bytes;
  const size_t gws_bytes = ws_bytes - w.bytes;
  const DerivedLayout L = derived_layout(d);
  const float *WcF = (const float *)derived + L.WcF;

  LFI_CUDA(cudaMemsetAsync(w.hstate, 0, (size_t)K * B * d.H * sizeof(float), st));
  if (w.cstate) LFI_CUDA(cudaMemsetAsync(w.cstate, 0, (size_t)K * B * d.H * sizeof(float), st));

  // the input projections of the encoders do not depend on the window: computed once (first chunk)
  for (int c0 = 0; c0 < Tgen; c0 += chunk) {
    const int Tc = (Tgen - c0 < chunk) ? (Tgen - c0) : chunk;
    const size_t Mc = (size_t)Tc * B;
    const int t0 = d.start_ts + c0;
    LFI_TRY(build_cond(s, d, p, bt, t0, Tc, w.cond, w.enc, w.gh, !teacher_forced, c0 == 0, gemm_mode, gws, gws_bytes, st));
    core::InvArgs a;
    memset(&a, 0, sizeof(a));
    a.d = d; a.dv = make_view(d, derived, p); a.B = B; a.Tc = Tc; a.k_hi = K - 1; a.k_lo = 0; a.g_k0 = 0;
    a.t_abs0 = t0; a.t_rel0 = c0; a.noise = noise;
    if (teacher_forced) {
      LFI_TRY(cond_to_gates(d, p, WcF, w.cond, Mc, w.Cs, w.G, gemm_mode, gws, gws_bytes, st));
      a.G = w.G; a.g_ld = (long)K * d.GH;
    } else {
      // static columns of cond_transform (pre-activation, bias included); the p1_face window is added in-kernel
      GemmArgs q = gemm_args(0, 1, (int)Mc, K * d.D, d.Fe - d.Far, w.cond + d.Far, d.Fe, WcF + d.Far, d.Fe, w.Cs, K * d.D,
                             LFI_EPI_BIAS, p->bc);
      if (d.Fe > d.Far) LFI_TRY(gemm_dispatch(gemm_mode, q, gws, gws_bytes, st));
      else LFI_TRY(aux::gather2d(w.Cs, K * d.D, p->bc, 0, 0, 1, 1, (int)Mc, K * d.D, st));  // no static modality: bias only
      a.cstatic = w.Cs; a.cs_ld = (long)K * d.D;
      a.faces = faces; a.f_sb = (long)seq_len * d.C; a.f_st = d.C;
    }
    a.faces_out = faces; a.fo_sb = (long)seq_len * d.C; a.fo_st = d.C;
    a.hstate = w.hstate; a.cstate = w.cstate; a.logdet_out = logdet_out;
    if (!teacher_forced && w.tc_ar) {
      // Tensor-core modes: the autoregressive part of the conditioning (p1_face window -> cond_transform -> gate-ih,
      // 340 k of the 410 k MAC per row and step) runs as two tcgen05 GEMMs per frame over all sequences; the persistent
      // kernel then walks the K inverse steps of that frame with the gate pre-activations given.  Still no host round
      // trip: everything is stream-ordered.
      const bool lo = gemm_mode == LFI_GEMM_BF16X3;
      const int In = d.Ci + d.D, hist0 = d.Far / d.C;
      if (c0 == 0) {  // operand planes of the two weights, once per call
        LFI_TRY(split_to_planes(WcF, K * d.D, d.Far, d.Fe, 0, 1, w.war_hi, lo ? w.war_lo : nullptr, st));
        LFI_TRY(split_to_planes(p->w_ih + d.Ci, d.GH, d.D, In, (long)d.GH * In, K, w.wihc_hi, lo ? w.wihc_lo : nullptr, st));
      }
      a.cstatic = nullptr; a.faces = nullptr;
      a.Tc = 1; a.G = w.G; a.g_ld = (long)K * d.GH;
      // The frame chain is ~6 short, strictly dependent launches per frame, issued directly: capturing a chunk of it into one
      // CUDA graph was measured on B200 (1,024 sequences x 750 frames) at 322.9 ms with and without the graph - the chain is
      // bound by the kernels themselves, not by launch gaps.
      for (int tc = 0; tc < Tc; ++tc) {
        LFI_TRY(aux::gather_windows(w.car, d.Far, 0, faces, nullptr, B, seq_len, d.C, hist0, 0, t0 + tc, 1, st));
        float *Cf = w.Cs + (size_t)tc * B * K * d.D;  // static pre-activation of this frame (bias included), updated in place
        GemmArgs q = gemm_args(0, 1, B, K * d.D, d.Far, w.car, d.Far, nullptr, d.Far, Cf, K * d.D, LFI_EPI_ACCUM_PRE | LFI_EPI_LRELU);
        q.pB = plane_ref(w.war_hi, w.war_lo, d.Far);
        q.pOut = plane_ref(w.cact_hi, w.cact_lo, K * d.D);
        LFI_TRY(gemm_dispatch(gemm_mode, q, gws, gws_bytes, st));
        GemmArgs h = gemm_args(0, 1, B, d.GH, d.D, nullptr, K * d.D, nullptr, d.D, w.G, K * d.GH, LFI_EPI_BIAS, p->b_ih);
        h.batch = K; h.sC = d.GH; h.sBias = d.GH;
        h.pA = plane_ref(w.cact_hi, w.cact_lo, K * d.D, d.D);
        h.pB = plane_ref(w.wihc_hi, w.wihc_lo, d.D, (long)d.GH * d.D);
        LFI_TRY(gemm_dispatch(gemm_mode, h, gws, gws_bytes, st));
        core::InvArgs af = a;
        af.t_abs0 = t0 + tc; af.t_rel0 = c0 + tc;
        LFI_TRY(core::launch_inv(af, st));
      }
      continue;
    }
    LFI_TRY(core::launch_inv(a, st));
  }
  return LFI_OK;
}

// ------------------------------------------------------------------------------------------------
// likelihood evaluation in chunks of frames: no stash, no gradients, the RNN state of the K flow steps carried between chunks
struct EvalWs {
  float *cond, *Cact, *G, *ld, *xin, *gh;
  void *cact_hi, *cact_lo;   // the cond_transform activations as operand planes (plan.planes), as in training
  float *hstate[2], *cstate[2];  // [K][B][H] carried state, ping-pong: chunk i reads slot i % 2 and leaves its final state in the other
  float *st_h, *st_c;        // Wave only: [K][chunk][B][H], the states the wavefront kernel passes between frames
  int *flags;
  EncWs enc[LFI_NMOD];
  core::CorePlan plan;
  size_t bytes;
};
// Everything but the encoders' input projections (plan_enc_nograd) is sized by the chunk, not by T.
static void plan_eval(const lfi_shape *s, const Dims &d, int B, int T, int chunk, int mode, void *ws, EvalWs *w) {
  Bump b(ws, 0);
  const size_t Mc = (size_t)chunk * B, K = d.K, KBH = K * B * d.H;
  w->plan = core::plan_core_eval(d, B, mode);
  const bool planes = w->plan.planes, wave = w->plan.fwd == core::CoreKernel::Wave;
  w->cond = b.take<float>(Mc * d.Fe);
  w->Cact = planes ? nullptr : b.take<float>(Mc * K * d.D);
  w->cact_hi = planes ? take_bf16(b, Mc * K * d.D) : nullptr;
  w->cact_lo = planes && mode == LFI_GEMM_BF16X3 ? take_bf16(b, Mc * K * d.D) : nullptr;
  w->G = b.take<float>(round_up_sz(Mc, 32) * K * d.GH);  // (whole 32-row blocks: the row-interleaved layout of the tensor-core core)
  w->ld = b.take<float>(Mc);
  w->xin = b.take<float>(K * Mc * d.C);
  w->flags = b.take<int>(kFlagInts);
  for (int i = 0; i < 2; ++i) {
    w->hstate[i] = b.take<float>(KBH);
    w->cstate[i] = d.G == 4 ? b.take<float>(KBH) : nullptr;
  }
  w->st_h = wave ? b.take<float>(K * Mc * d.H) : nullptr;
  w->st_c = wave && d.G == 4 ? b.take<float>(K * Mc * d.H) : nullptr;
  plan_enc_nograd(s, B, T, Mc, mode, b, w->enc, &w->gh);
  w->bytes = round_up_sz(b.off, 256);
}

size_t lfi_eval_ws_bytes(const lfi_shape *s, int B, int T, int chunk, int gemm_mode) {
  Dims d;
  if (make_dims(s, &d) != LFI_OK || B < 1 || chunk < 1 || T <= d.start_ts) return 0;
  chunk = std::min(chunk, T - d.start_ts);
  EvalWs w;
  plan_eval(s, d, B, T, chunk, gemm_mode, nullptr, &w);
  return w.bytes + gemm_scratch_bound(s, d, (size_t)chunk * B, (size_t)B * T, gemm_mode);
}

// SeqGlow.forward without gradients (models.py:534-561 under torch.no_grad()), chunk frames at a time: per chunk the conditioning
// (build_cond, the encoder paths of a call without gradients), the gate-ih pre-activations, then the forward flow core from the
// state the previous chunk left.  Stream-ordered throughout, no host round trip.
int lfi_seq_eval(const lfi_shape *s, const void *derived, const lfi_params *p, const lfi_batch *bt, int chunk, float *z,
                 float *nll, float *scale_out, void *ws, size_t ws_bytes, int gemm_mode, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  Dims d;
  LFI_TRY(make_dims(s, &d));
  LFI_REQUIRE(derived && p && bt && z && nll && ws, LFI_ERR_ARG, "lfi_seq_eval: null argument");
  LFI_REQUIRE(chunk >= 1, LFI_ERR_ARG, "lfi_seq_eval: chunk=%d must be >= 1", chunk);
  LFI_REQUIRE(bt->B >= 1 && bt->T > d.start_ts, LFI_ERR_ARG, "lfi_seq_eval: B=%d, T=%d (T must exceed the longest history %d)",
              bt->B, bt->T, d.start_ts);
  LFI_REQUIRE(bt->x[0], LFI_ERR_ARG, "lfi_seq_eval: batch: p1_face missing");
  const int B = bt->B, T = bt->T, Tp = T - d.start_ts, K = d.K;
  chunk = std::min(chunk, Tp);
  EvalWs w;
  plan_eval(s, d, B, T, chunk, gemm_mode, ws, &w);
  const size_t gneed = gemm_scratch_bound(s, d, (size_t)chunk * B, (size_t)B * T, gemm_mode);
  LFI_REQUIRE(ws_bytes >= w.bytes + gneed, LFI_ERR_WORKSPACE, "eval workspace too small: %zu < %zu", ws_bytes, w.bytes + gneed);
  void *gws = (char *)ws + w.bytes;
  const size_t gws_bytes = ws_bytes - w.bytes;
  const float *WcF = (const float *)derived + derived_layout(d).WcF;
  const bool wave = w.plan.fwd == core::CoreKernel::Wave;
  const size_t KBH = (size_t)K * B * d.H;

  LFI_CUDA(cudaMemsetAsync(w.hstate[0], 0, KBH * sizeof(float), st));  // models.py:196-202: state None = zeros
  if (w.cstate[0]) LFI_CUDA(cudaMemsetAsync(w.cstate[0], 0, KBH * sizeof(float), st));
  lfi_batch bc = *bt;
  for (int c0 = 0, cur = 0; c0 < Tp; c0 += chunk, cur ^= 1) {
    const int Tc = std::min(chunk, Tp - c0);
    const size_t Mc = (size_t)Tc * B;
    // the window kernels index the masks [T'][B][hist] by the window's index within the call
    for (int m = 0; m < LFI_NMOD; ++m) bc.mask[m] = bt->mask[m] ? bt->mask[m] + (size_t)c0 * B * s->hist[m] : nullptr;
    // (the input projections of the encoders do not depend on the window: computed once, on the first chunk)
    LFI_TRY(build_cond(s, d, p, &bc, d.start_ts + c0, Tc, w.cond, w.enc, w.gh, false, c0 == 0, gemm_mode, gws, gws_bytes, st));
    LFI_TRY(cond_to_gates(d, p, WcF, w.cond, Mc, w.Cact, w.G, gemm_mode, gws, gws_bytes, st, w.cact_hi, w.cact_lo, w.plan.tiled));
    core::FwdArgs a;
    memset(&a, 0, sizeof(a));
    a.d = d; a.dv = make_view(d, derived, p); a.B = B; a.Tp = Tc; a.k_first = 0; a.k_last = K - 1;
    a.x0 = bt->x[0] + (size_t)(d.start_ts + c0) * d.C; a.x_sb = (long)T * d.C; a.x_st = d.C;
    a.G = w.G; a.g_ld = (long)K * d.GH; a.g_k0 = 0;
    a.xin = w.xin; a.ld = w.ld; a.ld_accumulate = 0;
    a.nll = nll + (size_t)c0 * B; a.z_out = z + (size_t)c0 * B * d.C; a.scale_out = scale_out;
    a.flags = w.flags; a.flags_bytes = kFlagInts * sizeof(int);
    a.stash_tiled = a.g_tiled = w.plan.tiled ? 1 : 0;
    a.h0 = w.hstate[cur];
    if (wave) {
      a.c0 = w.cstate[cur]; a.st_h = w.st_h; a.st_c = w.st_c;
    } else {
      a.h_last = w.hstate[cur ^ 1];
    }
    LFI_TRY(core::launch_fwd(a, w.plan.fwd, st));
    if (wave && c0 + Tc < Tp) {  // the state after the chunk's last frame: cell (k, Tc - 1) of every step
      const size_t row = (size_t)B * d.H * sizeof(float), pitch = (size_t)Tc * row;
      LFI_CUDA(cudaMemcpy2DAsync(w.hstate[cur ^ 1], row, w.st_h + (size_t)(Tc - 1) * B * d.H, pitch, row, K, cudaMemcpyDeviceToDevice, st));
      if (w.st_c)
        LFI_CUDA(cudaMemcpy2DAsync(w.cstate[cur ^ 1], row, w.st_c + (size_t)(Tc - 1) * B * d.H, pitch, row, K, cudaMemcpyDeviceToDevice, st));
    }
  }
  return LFI_OK;
}

// ------------------------------------------------------------------------------------------------
// single frame, single step (module API)
size_t lfi_flowstep_ws_bytes(const lfi_shape *s, int B) {
  Dims d;
  if (make_dims(s, &d) != LFI_OK || B < 1) return 0;
  Bump b(nullptr, 0);
  b.take<float>((size_t)B * d.D);
  b.take<float>((size_t)B * d.GH);
  b.take<float>((size_t)B * d.C * 2);
  b.take<float>((size_t)B);
  return round_up_sz(b.off, 256) + 256;
}

}  // extern "C"

// lfi_flowstep; q (reverse direction only, lfi_flowstep_rev_fwd_train): also fill that stash.  The stash changes where the
// cond_transform output lives and which kernel instantiation runs, not what is computed.
static int flowstep_impl(const lfi_shape *s, const void *derived, const lfi_params *p, int k, int reverse, const float *x,
                         const float *cond, const float *h_in, const float *c_in, float *h_out, float *c_out, float *y,
                         float *logdet, float *scale_out, int B, void *ws, size_t ws_bytes, const StepStash *q, cudaStream_t st) {
  Dims d;
  LFI_TRY(make_dims(s, &d));
  LFI_REQUIRE(derived && p && x && cond && h_out && y && logdet && ws, LFI_ERR_ARG, "lfi_flowstep: null argument");
  LFI_REQUIRE(k >= 0 && k < d.K && B >= 1, LFI_ERR_ARG, "lfi_flowstep: bad step %d / batch %d", k, B);
  LFI_REQUIRE(d.G == 3 || c_out, LFI_ERR_ARG, "lfi_flowstep: LSTM needs c_out");
  LFI_REQUIRE(ws_bytes >= lfi_flowstep_ws_bytes(s, B), LFI_ERR_WORKSPACE, "flowstep workspace too small");
  Bump b(ws, ws_bytes);
  float *Cact = b.take<float>((size_t)B * d.D);
  if (q) Cact = q->Cact;
  float *G = b.take<float>((size_t)B * d.GH);
  float *xin = b.take<float>((size_t)B * d.C * 2);
  float *ldtmp = b.take<float>((size_t)B);
  void *gws = (char *)ws + round_up_sz(b.off, 256);
  const size_t gws_bytes = ws_bytes - round_up_sz(b.off, 256);
  const int In = d.Ci + d.D;
  // cond_transform with the raw (unfolded) feature vector, then the c-part of gate-ih
  GemmArgs g1 = gemm_args(0, 1, B, d.D, d.F, cond, d.F, p->wc + (size_t)k * d.D * d.F, d.F, Cact, d.D, LFI_EPI_BIAS | LFI_EPI_LRELU,
                          p->bc + (size_t)k * d.D);
  LFI_TRY(gemm_dispatch(LFI_GEMM_FP32, g1, gws, gws_bytes, st));
  GemmArgs g2 = gemm_args(0, 1, B, d.GH, d.D, Cact, d.D, p->w_ih + (size_t)k * d.GH * In + d.Ci, In, G, d.GH, LFI_EPI_BIAS,
                          p->b_ih + (size_t)k * d.GH);
  LFI_TRY(gemm_dispatch(LFI_GEMM_FP32, g2, gws, gws_bytes, st));
  const size_t koffH = (size_t)k * B * d.H;
  if (!reverse) {
    core::FwdArgs a;
    memset(&a, 0, sizeof(a));
    a.d = d; a.dv = make_view(d, derived, p); a.B = B; a.Tp = 1; a.k_first = k; a.k_last = k;
    a.x0 = x; a.x_sb = d.C; a.x_st = 0; a.G = G; a.g_ld = d.GH; a.g_k0 = k;
    a.h0 = h_in ? h_in - koffH : nullptr; a.c0 = c_in ? c_in - koffH : nullptr;
    a.xin = xin - (size_t)k * B * d.C;  // never touched for a single step, kept valid anyway
    a.st_h = h_out - koffH; a.st_c = c_out ? c_out - koffH : nullptr;
    a.ld = logdet; a.ld_accumulate = 1; a.nll = nullptr; a.z_out = y;
    a.scale_out = scale_out ? scale_out - (size_t)k * B * d.Cz : nullptr;
    return core::launch_fwd(a, core::CoreKernel::Wave, st);
  }
  // reverse: state is read and written in place by the persistent kernel
  if (h_in) LFI_CUDA(cudaMemcpyAsync(h_out, h_in, (size_t)B * d.H * sizeof(float), cudaMemcpyDeviceToDevice, st));
  else LFI_CUDA(cudaMemsetAsync(h_out, 0, (size_t)B * d.H * sizeof(float), st));
  if (d.G == 4) {
    if (c_in) LFI_CUDA(cudaMemcpyAsync(c_out, c_in, (size_t)B * d.H * sizeof(float), cudaMemcpyDeviceToDevice, st));
    else LFI_CUDA(cudaMemsetAsync(c_out, 0, (size_t)B * d.H * sizeof(float), st));
  }
  core::InvArgs a;
  memset(&a, 0, sizeof(a));
  a.d = d; a.dv = make_view(d, derived, p); a.B = B; a.Tc = 1; a.k_hi = k; a.k_lo = k; a.g_k0 = k;
  a.t_abs0 = 0; a.t_rel0 = 0; a.noise = x; a.G = G; a.g_ld = d.GH;
  a.faces_out = y; a.fo_sb = d.C; a.fo_st = 0;
  a.hstate = h_out - koffH; a.cstate = c_out ? c_out - koffH : nullptr;
  a.logdet_out = ldtmp;
  if (q) { a.st_x1 = q->y; a.st_zc = q->zf; a.st_gates = q->gates; a.st_ahn = d.G == 3 ? q->ahn : nullptr; a.st_o = q->o; }
  LFI_TRY(core::launch_inv(a, st));
  if (q) {
    LFI_CUDA(cudaMemcpyAsync(q->h, h_out, (size_t)B * d.H * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (d.G == 4) LFI_CUDA(cudaMemcpyAsync(q->c, c_out, (size_t)B * d.H * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  // logdet += (-sum log s) computed by the kernel
  LFI_TRY(aux::colsum(logdet, ldtmp, B, 1, B, 1.0f, st));
  return LFI_OK;
}

extern "C" {

int lfi_flowstep(const lfi_shape *s, const void *derived, const lfi_params *p, int k, int reverse, const float *x,
                 const float *cond, const float *h_in, const float *c_in, float *h_out, float *c_out, float *y,
                 float *logdet, float *scale_out, int B, void *ws, size_t ws_bytes, void *stream) {
  return flowstep_impl(s, derived, p, k, reverse, x, cond, h_in, c_in, h_out, c_out, y, logdet, scale_out, B, ws, ws_bytes, nullptr,
                       (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------
size_t lfi_invconv_ws_bytes(int K, int C) {
  const size_t n = (size_t)K * C * C;
  return 6 * round_up_sz(n * sizeof(float), 256) + round_up_sz(2 * n * sizeof(double), 256) + 256;
}

int lfi_invconv_compose(int K, int C, const float *pm, const float *l, const float *u, const float *log_s, const float *sign_s,
                        float *w, float *winv, void *ws, size_t ws_bytes, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  LFI_REQUIRE(pm && l && u && log_s && sign_s && w && ws, LFI_ERR_ARG, "lfi_invconv_compose: null argument");
  LFI_REQUIRE(C >= 1 && C <= 256 && K >= 1, LFI_ERR_SHAPE, "lfi_invconv_compose: C=%d K=%d", C, K);
  LFI_REQUIRE(ws_bytes >= lfi_invconv_ws_bytes(K, C), LFI_ERR_WORKSPACE, "invconv workspace too small");
  Bump b(ws, ws_bytes);
  const size_t n = (size_t)K * C * C;
  float *Lm = b.take<float>(n), *Um = b.take<float>(n), *T1 = b.take<float>(n), *Li = b.take<float>(n), *Ui = b.take<float>(n);
  double *scr = b.take<double>(2 * n);
  const long sM = (long)C * C;
  LFI_TRY(aux::lu_build(Lm, Um, l, u, log_s, sign_s, K, C, st));
  GemmArgs g = gemm_args(0, 0, C, C, C, Lm, C, Um, C, T1, C, 0);
  g.batch = K; g.sA = sM; g.sB = sM; g.sC = sM;
  LFI_TRY(gemm_simt(g, st));                                   // L U
  GemmArgs h = gemm_args(0, 0, C, C, C, pm, C, T1, C, w, C, 0);
  h.batch = K; h.sA = sM; h.sB = sM; h.sC = sM;
  LFI_TRY(gemm_simt(h, st));                                   // W = P (L U)
  if (winv) {
    LFI_TRY(aux::tri_inverse_f64(Li, Ui, scr, Lm, Um, K, C, st));
    GemmArgs q = gemm_args(0, 1, C, C, C, Li, C, pm, C, T1, C, 0);  // L^-1 P^-1,  P^-1 = P^T for a permutation
    q.batch = K; q.sA = sM; q.sB = sM; q.sC = sM;
    LFI_TRY(gemm_simt(q, st));
    GemmArgs r = gemm_args(0, 0, C, C, C, Ui, C, T1, C, winv, C, 0);  // U^-1 (L^-1 P^-1)
    r.batch = K; r.sA = sM; r.sB = sM; r.sC = sM;
    LFI_TRY(gemm_simt(r, st));
  }
  return LFI_OK;
}

int lfi_invconv_compose_bwd(int K, int C, const float *pm, const float *l, const float *u, const float *log_s,
                            const float *sign_s, const float *dw, float *dl, float *du, float *dlog_s, void *ws,
                            size_t ws_bytes, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  LFI_REQUIRE(pm && l && u && log_s && sign_s && dw && dl && du && dlog_s && ws, LFI_ERR_ARG, "lfi_invconv_compose_bwd: null argument");
  LFI_REQUIRE(ws_bytes >= lfi_invconv_ws_bytes(K, C), LFI_ERR_WORKSPACE, "invconv workspace too small");
  Bump b(ws, ws_bytes);
  const size_t n = (size_t)K * C * C;
  float *Lm = b.take<float>(n), *Um = b.take<float>(n), *T1 = b.take<float>(n), *dL = b.take<float>(n), *dU = b.take<float>(n);
  const long sM = (long)C * C;
  LFI_TRY(aux::lu_build(Lm, Um, l, u, log_s, sign_s, K, C, st));
  GemmArgs g = gemm_args(1, 0, C, C, C, pm, C, dw, C, T1, C, 0);   // T1 = P^T dW
  g.batch = K; g.sA = sM; g.sB = sM; g.sC = sM;
  LFI_TRY(gemm_simt(g, st));
  GemmArgs h = gemm_args(0, 1, C, C, C, T1, C, Um, C, dL, C, 0);   // dL = T1 U^T
  h.batch = K; h.sA = sM; h.sB = sM; h.sC = sM;
  LFI_TRY(gemm_simt(h, st));
  GemmArgs q = gemm_args(1, 0, C, C, C, Lm, C, T1, C, dU, C, 0);   // dU = L^T T1
  q.batch = K; q.sA = sM; q.sB = sM; q.sC = sM;
  LFI_TRY(gemm_simt(q, st));
  return aux::lu_mask_grads(dl, du, dlog_s, dL, dU, log_s, sign_s, K, C, st);
}

// ------------------------------------------------------------------------------------------------
int lfi_actnorm(const float *x, const float *bias, const float *logs, float *y, int B, int C, int reverse, void *stream) {
  LFI_REQUIRE(x && bias && logs && y && B >= 1 && C >= 1, LFI_ERR_ARG, "lfi_actnorm: bad argument");
  return aux::actnorm(x, bias, logs, y, B, C, reverse, (cudaStream_t)stream);
}

int lfi_matmul(const float *a, const float *bm, const float *bias, float *c, int M, int N, int Kd, int transB, void *stream) {
  LFI_REQUIRE(a && bm && c, LFI_ERR_ARG, "lfi_matmul: null argument");
  GemmArgs g = gemm_args(0, transB ? 1 : 0, M, N, Kd, a, Kd, bm, transB ? Kd : N, c, N, bias ? LFI_EPI_BIAS : 0, bias);
  return gemm_simt(g, (cudaStream_t)stream);
}

int lfi_nll(const float *z, const float *logdet, float *nll, int B, int C, void *stream) {
  LFI_REQUIRE(z && logdet && nll && B >= 1 && C >= 1, LFI_ERR_ARG, "lfi_nll: bad argument");
  return aux::nll(z, logdet, nll, B, C, (cudaStream_t)stream);
}

int lfi_expand_faces(const float *x, const float *means, const float *stds, size_t rows, int exp_dim, int jaw_dim, int neck_dim,
                     float *out, void *stream) {
  LFI_REQUIRE(x && out && (means != nullptr) == (stds != nullptr), LFI_ERR_ARG, "lfi_expand_faces: bad argument");
  LFI_REQUIRE(exp_dim >= 0 && jaw_dim >= 0 && neck_dim >= 0 && exp_dim <= 100 && jaw_dim <= 3 && neck_dim <= 3 && exp_dim + jaw_dim + neck_dim >= 1,
              LFI_ERR_SHAPE, "lfi_expand_faces: expression/jaw/neck = %d/%d/%d do not fit the 106-wide FLAME vector", exp_dim, jaw_dim, neck_dim);
  return aux::expand_faces(x, means, stds, rows, exp_dim, jaw_dim, neck_dim, out, (cudaStream_t)stream);
}

int lfi_gather_batch(const float *raw, const long long *row0, int B, int T, int dim, float *out, void *stream) {
  LFI_REQUIRE(raw && row0 && out && B >= 1 && T >= 1 && dim >= 1, LFI_ERR_ARG, "lfi_gather_batch: bad argument");
  return aux::gather_batch(raw, row0, B, T, dim, out, (cudaStream_t)stream);
}

int lfi_jerk(const float *x, int B, int T, int C, void *scratch8, float *out, void *stream) {
  LFI_REQUIRE(x && scratch8 && out && B >= 1 && C >= 1, LFI_ERR_ARG, "lfi_jerk: bad argument");
  LFI_REQUIRE(T >= 4, LFI_ERR_SHAPE, "lfi_jerk: a third difference needs T >= 4 frames (got %d)", T);
  LFI_REQUIRE(((uintptr_t)scratch8 & 7) == 0, LFI_ERR_ARG, "lfi_jerk: scratch must be 8-byte aligned");
  return aux::jerk(x, B, T, C, (double *)scratch8, out, (cudaStream_t)stream);
}

int lfi_clip_adam(float *theta, float *grad, float *m, float *v, size_t n, float lr, float beta1, float beta2, float eps,
                  float max_norm, float grad_scale, int step, float *norm_scratch, void *stream) {
  LFI_REQUIRE(theta && grad && m && v && norm_scratch && step >= 1, LFI_ERR_ARG, "lfi_clip_adam: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  LFI_TRY(aux::sumsq(norm_scratch, grad, n, st));
  return aux::clip_adam(theta, grad, m, v, n, lr, beta1, beta2, eps, max_norm, grad_scale, step, norm_scratch, st);
}

int lfi_clip_adam_dev(float *theta, float *grad, float *m, float *v, size_t n, const float *hyper, float beta1, float beta2, float eps,
                      float max_norm, float grad_scale, float *norm_scratch, void *stream) {
  LFI_REQUIRE(theta && grad && m && v && norm_scratch && hyper, LFI_ERR_ARG, "lfi_clip_adam_dev: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  LFI_TRY(aux::sumsq(norm_scratch, grad, n, st));
  return aux::clip_adam(theta, grad, m, v, n, 0.f, beta1, beta2, eps, max_norm, grad_scale, 1, norm_scratch, st, hyper);
}

int lfi_clip_sgd_dev(float *theta, float *grad, float *buf, size_t n, const float *hyper, float momentum, float dampening,
                     float weight_decay, int nesterov, float max_norm, float grad_scale, float *norm_scratch, void *stream) {
  LFI_REQUIRE(theta && grad && hyper && norm_scratch && n > 0, LFI_ERR_ARG, "lfi_clip_sgd_dev: bad argument");
  LFI_REQUIRE(momentum >= 0.f && weight_decay >= 0.f, LFI_ERR_ARG, "lfi_clip_sgd_dev: negative momentum or weight_decay");
  LFI_REQUIRE((buf != nullptr) == (momentum != 0.f), LFI_ERR_ARG, "lfi_clip_sgd_dev: buf must be given exactly when momentum != 0");
  LFI_REQUIRE(!nesterov || (momentum > 0.f && dampening == 0.f), LFI_ERR_ARG,
              "lfi_clip_sgd_dev: nesterov needs momentum > 0 and dampening 0");
  cudaStream_t st = (cudaStream_t)stream;
  LFI_TRY(aux::sumsq(norm_scratch, grad, n, st));
  return aux::clip_sgd(theta, grad, buf, n, hyper, momentum, dampening, weight_decay, nesterov ? 1 : 0, max_norm, grad_scale,
                       norm_scratch, st);
}

int lfi_clip_rmsprop_dev(float *theta, float *grad, float *square_avg, float *grad_avg, float *buf, size_t n, const float *hyper,
                         float alpha, float eps, float weight_decay, float momentum, float max_norm, float grad_scale,
                         float *norm_scratch, void *stream) {
  LFI_REQUIRE(theta && grad && square_avg && hyper && norm_scratch && n > 0, LFI_ERR_ARG, "lfi_clip_rmsprop_dev: bad argument");
  LFI_REQUIRE(alpha >= 0.f && eps >= 0.f && momentum >= 0.f && weight_decay >= 0.f, LFI_ERR_ARG,
              "lfi_clip_rmsprop_dev: negative alpha, eps, momentum or weight_decay");
  LFI_REQUIRE((buf != nullptr) == (momentum > 0.f), LFI_ERR_ARG, "lfi_clip_rmsprop_dev: buf must be given exactly when momentum > 0");
  cudaStream_t st = (cudaStream_t)stream;
  LFI_TRY(aux::sumsq(norm_scratch, grad, n, st));
  return aux::clip_rmsprop(theta, grad, square_avg, grad_avg, buf, n, hyper, alpha, eps, weight_decay, momentum, max_norm, grad_scale,
                           norm_scratch, st);
}

int lfi_gemm(int mode, int transA, int transB, int M, int N, int Kd, const float *A, int lda, long strideA, const float *Bm,
             int ldb, long strideB, float *Cm, int ldc, long strideC, const float *bias, long strideBias, const float *auxm,
             int ldaux, long strideAux, int batch, int epi, void *ws, size_t ws_bytes, void *stream) {
  GemmArgs g = gemm_args(transA, transB, M, N, Kd, A, lda, Bm, ldb, Cm, ldc, epi, bias);
  g.sA = strideA; g.sB = strideB; g.sC = strideC; g.sBias = strideBias; g.aux = auxm; g.ldaux = ldaux; g.sAux = strideAux;
  g.batch = batch;
  return gemm_dispatch(mode, g, ws, ws_bytes, (cudaStream_t)stream);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// FlowStep.forward with autograd (module API): forward with a stash (lfi_flowstep_rev_fwd_train: the reverse direction), and the
// backward of one cell (the reverse direction's backward, lfi_flowstep_rev_bwd, is in module_grad.cu).
extern "C" {

size_t lfi_flowstep_stash_bytes(const lfi_shape *s, int B) {
  Dims d;
  if (make_dims(s, &d) != LFI_OK || B < 1) return 0;
  StepStash q;
  plan_step_stash(d, B, nullptr, &q);
  return q.bytes;
}

size_t lfi_flowstep_bwd_ws_bytes(const lfi_shape *s, int B) {
  Dims d;
  if (make_dims(s, &d) != LFI_OK || B < 1) return 0;
  Bump b(nullptr, 0);
  b.take<float>((size_t)B * d.GH);  // dG
  b.take<float>((size_t)B * d.GH);  // dAh
  b.take<float>((size_t)B * d.Co);  // dO
  b.take<float>((size_t)B * d.C);   // dzf
  b.take<float>((size_t)B * d.D);   // dCact
  return round_up_sz(b.off, 256) + 256;
}

int lfi_flowstep_fwd_train(const lfi_shape *s, const void *derived, const lfi_params *p, int k, const float *x, const float *cond,
                           const float *h_in, const float *c_in, float *h_out, float *c_out, float *y, float *logdet,
                           float *scale_out, int B, void *stash, size_t stash_bytes, void *ws, size_t ws_bytes, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  Dims d;
  LFI_TRY(make_dims(s, &d));
  LFI_REQUIRE(derived && p && x && cond && h_out && y && logdet && ws && stash, LFI_ERR_ARG, "lfi_flowstep_fwd_train: null argument");
  LFI_REQUIRE(k >= 0 && k < d.K && B >= 1, LFI_ERR_ARG, "lfi_flowstep_fwd_train: bad step %d / batch %d", k, B);
  LFI_REQUIRE(d.G == 3 || c_out, LFI_ERR_ARG, "lfi_flowstep_fwd_train: LSTM needs c_out");
  StepStash q;
  plan_step_stash(d, B, stash, &q);
  LFI_REQUIRE(stash_bytes >= q.bytes, LFI_ERR_WORKSPACE, "flowstep stash too small: %zu < %zu", stash_bytes, q.bytes);
  LFI_REQUIRE(ws_bytes >= lfi_flowstep_ws_bytes(s, B), LFI_ERR_WORKSPACE, "flowstep workspace too small");
  Bump b(ws, ws_bytes);
  b.take<float>((size_t)B * d.D);
  float *G = b.take<float>((size_t)B * d.GH);
  float *xin = b.take<float>((size_t)B * d.C * 2);
  void *gws = (char *)ws + round_up_sz(b.off, 256);
  const size_t gws_bytes = ws_bytes - round_up_sz(b.off, 256);
  const int In = d.Ci + d.D;
  GemmArgs g1 = gemm_args(0, 1, B, d.D, d.F, cond, d.F, p->wc + (size_t)k * d.D * d.F, d.F, q.Cact, d.D, LFI_EPI_BIAS | LFI_EPI_LRELU,
                          p->bc + (size_t)k * d.D);
  LFI_TRY(gemm_dispatch(LFI_GEMM_FP32, g1, gws, gws_bytes, st));
  GemmArgs g2 = gemm_args(0, 1, B, d.GH, d.D, q.Cact, d.D, p->w_ih + (size_t)k * d.GH * In + d.Ci, In, G, d.GH, LFI_EPI_BIAS,
                          p->b_ih + (size_t)k * d.GH);
  LFI_TRY(gemm_dispatch(LFI_GEMM_FP32, g2, gws, gws_bytes, st));
  const size_t kB = (size_t)k * B;
  core::FwdArgs a;
  memset(&a, 0, sizeof(a));
  a.d = d; a.dv = make_view(d, derived, p); a.B = B; a.Tp = 1; a.k_first = k; a.k_last = k;
  a.x0 = x; a.x_sb = d.C; a.x_st = 0; a.G = G; a.g_ld = d.GH; a.g_k0 = k;
  a.h0 = h_in ? h_in - kB * d.H : nullptr; a.c0 = c_in ? c_in - kB * d.H : nullptr;
  a.xin = xin - kB * d.C;
  // the stash arrays are [K][Tp][B][width]: moved back by k cells so that cell (k, 0) lands on the caller's buffers
  a.st_y = q.y - kB * d.C; a.st_zf = q.zf - kB * d.C; a.st_h = q.h - kB * d.H; a.st_c = d.G == 4 ? q.c - kB * d.H : nullptr;
  a.st_gates = q.gates - kB * d.GH; a.st_ahn = d.G == 3 ? q.ahn - kB * d.H : nullptr; a.st_o = q.o - kB * d.Co;
  a.ld = logdet; a.ld_accumulate = 1; a.nll = nullptr; a.z_out = y;
  a.scale_out = scale_out ? scale_out - kB * d.Cz : nullptr;
  LFI_TRY(core::launch_fwd(a, core::CoreKernel::Wave, st));
  LFI_CUDA(cudaMemcpyAsync(h_out, q.h, (size_t)B * d.H * sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (d.G == 4) LFI_CUDA(cudaMemcpyAsync(c_out, q.c, (size_t)B * d.H * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return LFI_OK;
}

int lfi_flowstep_rev_fwd_train(const lfi_shape *s, const void *derived, const lfi_params *p, int k, const float *x, const float *cond,
                               const float *h_in, const float *c_in, float *h_out, float *c_out, float *y, float *logdet, int B,
                               void *stash, size_t stash_bytes, void *ws, size_t ws_bytes, void *stream) {
  Dims d;
  LFI_TRY(make_dims(s, &d));
  LFI_REQUIRE(stash, LFI_ERR_ARG, "lfi_flowstep_rev_fwd_train: null stash");
  LFI_REQUIRE(B >= 1, LFI_ERR_ARG, "lfi_flowstep_rev_fwd_train: bad batch %d", B);
  StepStash q;
  plan_step_stash(d, B, stash, &q);
  LFI_REQUIRE(stash_bytes >= q.bytes, LFI_ERR_WORKSPACE, "flowstep stash too small: %zu < %zu", stash_bytes, q.bytes);
  return flowstep_impl(s, derived, p, k, 1, x, cond, h_in, c_in, h_out, c_out, y, logdet, nullptr, B, ws, ws_bytes, &q,
                       (cudaStream_t)stream);
}

int lfi_flowstep_bwd(const lfi_shape *s, const void *derived, const lfi_params *p, int k, const float *cond, const float *h_in,
                     const float *c_in, const float *dy, const float *dlogdet, const float *dh_out, const float *dc_out, float *dx,
                     float *dcond, float *dh_in, float *dc_in, lfi_params *g, int B, void *stash, size_t stash_bytes, void *ws,
                     size_t ws_bytes, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  Dims d;
  LFI_TRY(make_dims(s, &d));
  LFI_REQUIRE(derived && p && cond && dy && dx && dcond && dh_in && g && stash && ws, LFI_ERR_ARG, "lfi_flowstep_bwd: null argument");
  LFI_REQUIRE(k >= 0 && k < d.K && B >= 1, LFI_ERR_ARG, "lfi_flowstep_bwd: bad step %d / batch %d", k, B);
  LFI_REQUIRE(d.G == 3 || dc_in, LFI_ERR_ARG, "lfi_flowstep_bwd: LSTM needs dc_in");
  StepStash q;
  plan_step_stash(d, B, stash, &q);
  LFI_REQUIRE(stash_bytes >= q.bytes, LFI_ERR_WORKSPACE, "flowstep stash too small");
  LFI_REQUIRE(ws_bytes >= lfi_flowstep_bwd_ws_bytes(s, B), LFI_ERR_WORKSPACE, "flowstep backward workspace too small");
  Bump b(ws, ws_bytes);
  float *dG = b.take<float>((size_t)B * d.GH), *dAh = b.take<float>((size_t)B * d.GH), *dO = b.take<float>((size_t)B * d.Co);
  float *dzf = b.take<float>((size_t)B * d.C), *dC = b.take<float>((size_t)B * d.D);
  const int C = d.C, Ci = d.Ci, GH = d.GH, H = d.H, D = d.D, Co = d.Co, In = Ci + D, F = d.F;
  const size_t kB = (size_t)k * B;
  core::BwdArgs a;
  memset(&a, 0, sizeof(a));
  a.d = d; a.dv = make_view(d, derived, p); a.B = B; a.Tp = 1; a.single = k;
  a.st.y = q.y - kB * C; a.st.zf = q.zf - kB * C; a.st.h = q.h - kB * H; a.st.c = d.G == 4 ? q.c - kB * H : nullptr;
  a.st.gates = q.gates - kB * GH; a.st.ahn = d.G == 3 ? q.ahn - kB * H : nullptr; a.st.o = q.o - kB * Co;
  a.dz_ext = dy; a.dld_ext = dlogdet; a.dh_ext = dh_out; a.dc_ext = dc_out; a.h_prev_ext = h_in; a.c_prev_ext = c_in;
  a.dx0_out = dx; a.dh0_out = dh_in; a.dc0_out = dc_in;
  a.dG = dG; a.dg_ld = GH; a.dg_k0 = k;
  a.dAh = dAh - kB * GH; a.dO = dO - kB * Co; a.dzf = dzf - kB * C;
  a.g_an_bias = g->an_bias; a.g_an_logs = g->an_logs; a.g_b_hh = g->b_hh; a.g_bf = g->bf; a.g_lf = g->lf;
  LFI_TRY(core::launch_bwd_single(a, st));
  // weight gradients of this cell (fp32 tiles): reductions over the B rows
  auto wg = [&](int Mo, int No, const float *A, int lda, const float *Bm, int ldb, float *Cm, int ldc) -> int {
    GemmArgs r = gemm_args(1, 0, Mo, No, B, A, lda, Bm, ldb, Cm, ldc, LFI_EPI_ACCUM);
    return gemm_simt(r, st);
  };
  if (h_in) LFI_TRY(wg(GH, H, dAh, GH, h_in, H, g->w_hh + (size_t)k * GH * H, H));
  LFI_TRY(wg(GH, Ci, dG, GH, q.zf, C, g->w_ih + (size_t)k * GH * In, In));
  LFI_TRY(wg(GH, D, dG, GH, q.Cact, D, g->w_ih + (size_t)k * GH * In + Ci, In));
  LFI_TRY(wg(Co, H, dO, Co, q.h, H, g->wf + (size_t)k * Co * H, H));
  LFI_TRY(wg(C, C, q.y, C, dzf, C, g->w + (size_t)k * C * C, C));
  LFI_TRY(aux::colsum(g->b_ih + (size_t)k * GH, dG, GH, B, GH, 1.0f, st));
  // cond_transform backward: dC = (dG W_ih[:, Ci:]) * LeakyReLU'(Cact); d b_c, d W_c, d cond
  GemmArgs t = gemm_args(0, 0, B, D, GH, dG, GH, p->w_ih + (size_t)k * GH * In + Ci, In, dC, D, LFI_EPI_LRELU_BWD);
  t.aux = q.Cact; t.ldaux = D;
  LFI_TRY(gemm_simt(t, st));
  LFI_TRY(aux::colsum(g->bc + (size_t)k * D, dC, D, B, D, 1.0f, st));
  LFI_TRY(wg(D, F, dC, D, cond, F, g->wc + (size_t)k * D * F, F));
  GemmArgs u = gemm_args(0, 0, B, F, D, dC, D, p->wc + (size_t)k * D * F, F, dcond, F, 0);
  LFI_TRY(gemm_simt(u, st));
  return LFI_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// FeatureEncoder / ModalityEncoder.forward with autograd (module API): the window GRUs with the training step's per-step launches
// and stash, and their backward with written, bit-reproducible gradients and the gradient of the raw streams.
namespace lfi {
struct FeatPlan {
  EncWs enc[LFI_NMOD];
  float *gh;                  // forward: [M][3E] recurrent products of the unfused window steps
  float *part, *dxg;          // backward: bias-gradient partials and dXg of the largest modality (modalities run one after another)
  int part_rows[LFI_NMOD];
  size_t stash_bytes, ws_bytes;  // (ws_bytes: the call's workspace before its GEMM scratch)
};
// The stash layout depends on (shape, B, Tp, mode) only, so the forward and the backward call find the same arrays in it.
static void plan_feature(const lfi_shape *s, int B, int T, int Tp, int mode, void *stash, void *ws, bool bwd, FeatPlan *f) {
  Bump S(stash, 0), W(ws, 0), none(nullptr, 0);
  const EncBumps eb = {&S, bwd ? &none : &W, &W, bwd ? &W : &none};
  const size_t M = (size_t)Tp * B;
  size_t ghmax = 0, partmax = 0, xgmax = 0;
  for (int m = 0; m < LFI_NMOD; ++m) {
    memset(&f->enc[m], 0, sizeof(EncWs));
    f->part_rows[m] = 0;
    if (s->hist[m] <= 0 || s->ehid[m] <= 0) continue;
    const size_t E = s->ehid[m];
    plan_enc_train(s, m, B, T, M, mode, eb, f->enc[m]);
    f->part_rows[m] = aux::enc_gate_bwd2_part_rows((int)M, (int)E);
    ghmax = ghmax > M * 3 * E ? ghmax : M * 3 * E;
    partmax = partmax > f->part_rows[m] * 4 * E ? partmax : f->part_rows[m] * 4 * E;
    xgmax = xgmax > s->hist[m] * M * s->dim[m] ? xgmax : s->hist[m] * M * s->dim[m];
  }
  f->gh = bwd ? nullptr : W.take<float>(ghmax);
  f->part = bwd ? W.take<float>(partmax) : nullptr;
  f->dxg = bwd ? W.take<float>(xgmax) : nullptr;
  f->stash_bytes = round_up_sz(S.off, 256);
  f->ws_bytes = round_up_sz(W.off, 256);
}

// Operand-plane scratch of the backward GEMMs: only modalities whose encoder does not run on operand planes split fp32 operands.
static size_t feature_bwd_scratch(const lfi_shape *s, const FeatPlan &f, int Tp, int B, int mode) {
  size_t need = 0;
  const int M = Tp * B;
  for (int m = 0; m < LFI_NMOD; ++m) {
    if (s->hist[m] <= 0 || s->ehid[m] <= 0 || f.enc[m].plan.planes) continue;
    const int E = s->ehid[m], dim = s->dim[m], h = s->hist[m];
    const GemmArgs gs[] = {gemm_args(0, 0, M, E, 3 * E, nullptr, 3 * E, nullptr, E, nullptr, E),
                           gemm_args(1, 0, 3 * E, E, (h - 1) * M, nullptr, 3 * E, nullptr, E, nullptr, E),
                           gemm_args(1, 0, 2 * E, dim, h * M, nullptr, 3 * E, nullptr, dim, nullptr, dim),
                           gemm_args(0, 0, h * M, dim, 2 * E, nullptr, 3 * E, nullptr, dim, nullptr, dim)};
    for (const GemmArgs &g : gs) need = need > gemm_ws_bytes_for(mode, g) ? need : gemm_ws_bytes_for(mode, g);
  }
  return need;
}
static size_t feature_fwd_need(const lfi_shape *s, const Dims &d, int B, int T, int Tp, int mode) {
  FeatPlan f;
  plan_feature(s, B, T, Tp, mode, nullptr, nullptr, false, &f);
  return f.ws_bytes + gemm_scratch_bound(s, d, (size_t)Tp * B, (size_t)B * T, mode);
}
static size_t feature_bwd_need(const lfi_shape *s, int B, int T, int Tp, int mode) {
  FeatPlan f;
  plan_feature(s, B, T, Tp, mode, nullptr, nullptr, true, &f);
  return f.ws_bytes + feature_bwd_scratch(s, f, Tp, B, mode);
}

// One workspace size serves both calls (lfi_feature_bwd_ws_bytes).
static size_t feature_ws_need(const lfi_shape *s, const Dims &d, int B, int T, int Tp, int mode) {
  const size_t a = feature_fwd_need(s, d, B, T, Tp, mode), b = feature_bwd_need(s, B, T, Tp, mode);
  return a > b ? a : b;
}

static int feature_train_dims(const lfi_shape *s, int B, int Tp, int mode, Dims *d) {
  LFI_TRY(make_dims(s, d));
  LFI_REQUIRE(s->f_raw <= 0, LFI_ERR_SHAPE, "feature encoder: the shape has no encoders (f_raw = %d)", s->f_raw);
  LFI_REQUIRE(B >= 1 && Tp >= 1, LFI_ERR_SHAPE, "feature encoder: B=%d Tp=%d must be >= 1", B, Tp);
  LFI_REQUIRE(mode >= LFI_GEMM_FP32 && mode <= LFI_GEMM_BF16, LFI_ERR_ARG, "feature encoder: unknown gemm mode %d", mode);
  return LFI_OK;
}

// Arguments both calls share: frames inside the batch, every stream the shape names present, the GRU weights (and gradients) set.
static int feature_check(const lfi_shape *s, const Dims &d, const lfi_params *p, const lfi_batch *bt, int t0, int Tp, const lfi_params *g,
                         const char *what) {
  LFI_REQUIRE(t0 >= d.start_ts && t0 + Tp <= bt->T, LFI_ERR_SHAPE, "%s: frames [%d,%d) outside [%d,%d)", what, t0, t0 + Tp, d.start_ts, bt->T);
  for (int m = 0; m < LFI_NMOD; ++m) {
    if (s->hist[m] <= 0) continue;
    LFI_REQUIRE(bt->x[m], LFI_ERR_ARG, "%s: batch modality %d missing", what, m);
    if (s->ehid[m] <= 0) continue;
    LFI_REQUIRE(p->enc_w_ih[m] && p->enc_w_hh[m] && p->enc_b_ih[m] && p->enc_b_hh[m], LFI_ERR_ARG, "%s: encoder %d weights missing", what, m);
    LFI_REQUIRE(!g || (g->enc_w_ih[m] && g->enc_w_hh[m] && g->enc_b_ih[m] && g->enc_b_hh[m]), LFI_ERR_ARG,
                "%s: encoder %d gradients missing", what, m);
  }
  return LFI_OK;
}
}  // namespace lfi

extern "C" {

size_t lfi_feature_stash_bytes(const lfi_shape *s, int B, int T, int Tp, int gemm_mode) {
  Dims d;
  if (feature_train_dims(s, B, Tp, gemm_mode, &d) != LFI_OK) return 0;
  FeatPlan f;
  plan_feature(s, B, T, Tp, gemm_mode, nullptr, nullptr, false, &f);
  return f.stash_bytes;
}

size_t lfi_feature_bwd_ws_bytes(const lfi_shape *s, int B, int T, int Tp, int gemm_mode) {
  Dims d;
  if (feature_train_dims(s, B, Tp, gemm_mode, &d) != LFI_OK) return 0;
  return feature_ws_need(s, d, B, T, Tp, gemm_mode);
}

int lfi_feature_encode_fwd_train(const lfi_shape *s, const lfi_params *p, const lfi_batch *bt, int t0, int Tp, float *cond, void *stash,
                                 size_t stash_bytes, void *ws, size_t ws_bytes, int gemm_mode, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  LFI_REQUIRE(s && p && bt && cond && stash && ws, LFI_ERR_ARG, "lfi_feature_encode_fwd_train: null argument");
  Dims d;
  LFI_TRY(feature_train_dims(s, bt->B, Tp, gemm_mode, &d));
  LFI_TRY(feature_check(s, d, p, bt, t0, Tp, nullptr, "lfi_feature_encode_fwd_train"));
  FeatPlan f;
  plan_feature(s, bt->B, bt->T, Tp, gemm_mode, stash, ws, false, &f);
  LFI_REQUIRE(stash_bytes >= f.stash_bytes, LFI_ERR_WORKSPACE, "lfi_feature_encode_fwd_train: stash too small: %zu < %zu", stash_bytes,
              f.stash_bytes);
  const size_t need = feature_ws_need(s, d, bt->B, bt->T, Tp, gemm_mode);
  LFI_REQUIRE(ws_bytes >= need, LFI_ERR_WORKSPACE, "lfi_feature_encode_fwd_train: workspace too small: %zu < %zu", ws_bytes, need);
  return build_cond(s, d, p, bt, t0, Tp, cond, f.enc, f.gh, false, true, gemm_mode, (char *)ws + f.ws_bytes, ws_bytes - f.ws_bytes, st);
}

int lfi_feature_encode_bwd(const lfi_shape *s, const lfi_params *p, const lfi_batch *bt, int t0, int Tp, const float *dcond,
                           float *const dx[LFI_NMOD], lfi_params *g, void *stash, size_t stash_bytes, void *ws, size_t ws_bytes,
                           int gemm_mode, void *stream) {
  cudaStream_t st = (cudaStream_t)stream;
  LFI_REQUIRE(s && p && bt && dcond && g && stash && ws, LFI_ERR_ARG, "lfi_feature_encode_bwd: null argument");
  Dims d;
  LFI_TRY(feature_train_dims(s, bt->B, Tp, gemm_mode, &d));
  LFI_TRY(feature_check(s, d, p, bt, t0, Tp, g, "lfi_feature_encode_bwd"));
  const int B = bt->B, T = bt->T;
  FeatPlan f;
  plan_feature(s, B, T, Tp, gemm_mode, stash, ws, true, &f);
  LFI_REQUIRE(stash_bytes >= f.stash_bytes, LFI_ERR_WORKSPACE, "lfi_feature_encode_bwd: stash too small: %zu < %zu", stash_bytes, f.stash_bytes);
  const size_t need = feature_ws_need(s, d, B, T, Tp, gemm_mode);
  LFI_REQUIRE(ws_bytes >= need, LFI_ERR_WORKSPACE, "lfi_feature_encode_bwd: workspace too small: %zu < %zu", ws_bytes, need);
  void *gws = (char *)ws + f.ws_bytes;
  const size_t gws_bytes = ws_bytes - f.ws_bytes;
  const bool lo = gemm_mode == LFI_GEMM_BF16X3;
  for (int m = 0; m < LFI_NMOD; ++m) {
    if (s->hist[m] <= 0) continue;
    float *dxm = dx ? dx[m] : nullptr;
    const int hist = s->hist[m], dim = s->dim[m], E = s->ehid[m];
    if (E <= 0) {  // "enc: none": the window itself is the feature block
      if (dxm) LFI_TRY(aux::window_grad(dxm, dcond + d.enc_offe[m], d.Fe, 0, bt->mask[m], B, T, dim, hist, m == 0 ? 0 : 1, t0, Tp, st));
      continue;
    }
    EncWs &ew = f.enc[m];
    if (ew.plan.planes) {  // the operand planes of W_hh (dh_prev) and W_ih (dXg) belong to this call's workspace
      LFI_TRY(split_to_planes(p->enc_w_hh[m], 3 * E, E, E, 0, 1, ew.whh_hi, lo ? ew.whh_lo : nullptr, st));
      if (dxm) LFI_TRY(split_to_planes(p->enc_w_ih[m], 3 * E, dim, dim, 0, 1, ew.wih_hi, lo ? ew.wih_lo : nullptr, st));
    }
    const EncBwdOpts o = {f.part, f.part_rows[m], f.dxg, dxm};
    LFI_TRY(enc_bwd(s, d, p, bt, t0, Tp, m, ew, dcond, g, gemm_mode, gemm_mode, gws, gws_bytes, o, st));
  }
  return LFI_OK;
}

}  // extern "C"
