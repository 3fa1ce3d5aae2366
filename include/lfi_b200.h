/*
 * lfi_b200.h — C ABI of the B200-native conditional-Glow hot path ("Let's Face It" MoGlow flow).
 *
 * The reference (jonepatr/lets_face_it) has no FFI layer: the path sits behind the Python module
 * API of code/glow_pytorch/glow/{models,modules}.py.  These entry points are what a binding for
 * that API binds (ctypes stub: lets_face_it_b200/_cabi.py; see INTEGRATION.md).  Every function
 *   - takes plain device pointers + sizes + a cudaStream_t (as void*), borrows them for the call,
 *   - allocates nothing (the caller passes a workspace sized by the matching *_ws_bytes call),
 *   - is stream-ordered, not thread-safe (the reference modules are stateful, SURVEY.md §8(b)),
 *   - returns 0 on success, a negative lfi_status otherwise; lfi_last_error() gives the text.
 * All tensors are contiguous fp32 unless stated.  Row index of every "[M, ...]" matrix is
 * m = t'*B + b (frame-major), t' = t - start_ts.
 */
#ifndef LFI_B200_H
#define LFI_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LFI_ABI_VERSION 11
#define LFI_NMOD 4 /* p1_face, p2_face, p1_speech, p2_speech — concat order of models.py:127-145 */

typedef enum lfi_status {
  LFI_OK = 0,
  LFI_ERR_SHAPE = -1,   /* unsupported / inconsistent shape */
  LFI_ERR_CUDA = -2,    /* a CUDA runtime call or launch failed */
  LFI_ERR_ARG = -3,     /* null / misaligned pointer, bad flag */
  LFI_ERR_WORKSPACE = -4 /* workspace too small */
} lfi_status;

/* GEMM numerics for the time-parallel contractions (cond_transform, gate-ih, encoders, wgrads). */
typedef enum lfi_gemm_mode {
  LFI_GEMM_FP32 = 0,       /* fp32 FFMA tiles (exact reference semantics)                       */
  LFI_GEMM_BF16X3 = 1,     /* tcgen05 bf16 tiles, 3-product split (a_hi b_hi + a_hi b_lo + a_lo b_hi): fp32-grade */
  LFI_GEMM_BF16 = 2        /* tcgen05 bf16 tiles, single product (throughput mode, looser bound) */
} lfi_gemm_mode;

/* Shapes of one model (final_model.yaml: C=56 K=16 H=128 D=512 G=3). */
typedef struct lfi_shape {
  int32_t C;              /* flow channels = Conditioning.p1_face.dim (models.py:473)            */
  int32_t K;              /* flow steps K*L (models.py:417-436)                                   */
  int32_t H;              /* coupling RNN hidden = Glow.hidden_channels, multiple of 4            */
  int32_t D;              /* Conditioning.cond_dim                                                */
  int32_t G;              /* gates: 3 = GRUCell (r,z,n), 4 = LSTMCell (i,f,g,o) (models.py:176-185) */
  int32_t affine;         /* 1 = affine coupling, 0 = additive (models.py:331-341)                */
  float scale_eps;        /* Glow.scale_eps: sigmoid(.+2).clamp(scale_eps)                        */
  int32_t hist[LFI_NMOD]; /* history per modality, 0 = modality absent (never for p1_face)        */
  int32_t dim[LFI_NMOD];  /* raw feature dim per modality                                         */
  int32_t ehid[LFI_NMOD]; /* GRU encoder hidden ("enc: rnn"), 0 = "enc: none" (flattened window)  */
  int32_t f_raw;          /* > 0: no FeatureEncoder, conditioning is a raw [B, f_raw] matrix (stand-alone
                             FlowStep / FlowNet as in test_modules.py:30-67); hist/dim/ehid are ignored and only
                             lfi_derive / lfi_flowstep are valid                                           */
} lfi_shape;

/* Trainable parameters, as [K, ...] blocks (flat storage, state-dict views live on top of it). */
typedef struct lfi_params {
  float *an_bias, *an_logs;          /* [K,C]      layers.k.actnorm.{bias,logs}  (modules.py:22-23)       */
  float *w;                          /* [K,C,C]    composed 1x1 weight W (modules.py:163-173), z = x @ W   */
  float *wc, *bc;                    /* [K,D,F],[K,D]  layers.k.f.cond_transform.0.{weight,bias}           */
  float *w_ih, *b_ih;                /* [K,G*H,C/2+D],[K,G*H]  layers.k.f.rnn.{weight_ih,bias_ih}          */
  float *w_hh, *b_hh;                /* [K,G*H,H],[K,G*H]      layers.k.f.rnn.{weight_hh,bias_hh}          */
  float *wf, *bf, *lf;               /* [K,Co,H],[K,Co],[K,Co] layers.k.f.final_linear.{weight,bias,logs}  */
  float *enc_w_ih[LFI_NMOD];         /* [3E,d]  feature_encoder.<m>_encoder.encoder.weight_ih_l0 (NULL if none) */
  float *enc_w_hh[LFI_NMOD];         /* [3E,E]                                    weight_hh_l0             */
  float *enc_b_ih[LFI_NMOD];         /* [3E]                                      bias_ih_l0               */
  float *enc_b_hh[LFI_NMOD];         /* [3E]                                      bias_hh_l0               */
} lfi_params;

/* One batch: models.py:534-559 reads batch[m][:, t-h+1 : t+1]; tensors are [B, T, dim[m]] batch-first
 * (mimicry_data_module.py layout).  mask[m] is NULL or the dropout mask [T', B, hist[m]] already
 * scaled by 1/(1-p) (models.py:56-58). */
typedef struct lfi_batch {
  const float *x[LFI_NMOD];
  const float *mask[LFI_NMOD];
  int32_t B, T;
} lfi_batch;

const char *lfi_last_error(void);
int lfi_abi_version(void);
long lfi_launch_count(void); /* kernels launched by this library since load (bench.py gpu_launches) */
/* Data-parallel hook (SURVEY.md section 8(e): the one exchange of the path is the gradient all-reduce after
 * LetsFaceItGlow.training_step's backward, lets_face_it_glow.py:39-59).  When an event (cudaEvent_t) is set, the next
 * lfi_seq_train_bwd records it on its stream as soon as the gradients of the flow-step weights (wc, bc, w_ih, b_ih, w_hh,
 * b_hh, wf, bf, lf) are final, i.e. before the encoder backward: the caller can start reducing that bucket while the
 * rest of the call runs.  NULL clears the hook. */
int lfi_set_grad_ready_event(void *event);

/* Optional overlap hook of the training forward: `event` (cudaEvent_t) marks the derived cache `derived` (lfi_invconv_compose +
 * lfi_derive, a chain of ~25 short launches per step) as rebuilt on ANOTHER stream.  While it is set, lfi_seq_train_fwd runs the
 * conditioning encoders - which read their parameters directly - first and waits for the event only in front of the first
 * consumer of the cache (the cond_transform GEMM), so the rebuild hides behind the encoder forward.  NULL clears the hook. */
int lfi_set_derived_ready_event(void *event);

/* ---- sizes ------------------------------------------------------------------------------- */
int lfi_feature_dim(const lfi_shape *s);        /* F  = FeatureEncoder.dim (models.py:96-125)            */
int lfi_feature_dim_folded(const lfi_shape *s); /* Fe = F with duplicated GRU halves folded (models.py:64) */
int lfi_start_ts(const lfi_shape *s);           /* utils.py:44-50                                        */
int lfi_coupling_out(const lfi_shape *s);       /* Co: f_seq output channels (models.py:276-298)         */
size_t lfi_derived_bytes(const lfi_shape *s);
size_t lfi_train_ws_bytes(const lfi_shape *s, int B, int T, int gemm_mode);
size_t lfi_sample_ws_bytes(const lfi_shape *s, int B, int T, int chunk, int gemm_mode);
size_t lfi_invconv_ws_bytes(int K, int C);
/* operand-plane scratch lfi_gemm needs for one problem in the tensor-core modes (0 in fp32 mode); the *_ws_bytes
 * functions above already include the scratch of the GEMMs they run */
size_t lfi_gemm_ws_bytes(int mode, int transA, int transB, int M, int N, int K, int batch);

/* ---- derived weight cache (transposes, folded cond_transform, padded slices, W^-1) --------
 * Must be re-run after every parameter update.  winv may be NULL (training only). */
int lfi_derive(const lfi_shape *s, const lfi_params *p, const float *winv, void *derived, int gemm_mode,
               void *stream);

/* ---- 1x1 conv LU parametrisation (modules.py:149-178) ------------------------------------- */
/* W = P (L*mask+I)(U*mask^T + diag(sign_s e^{log_s})) per step;  winv = U^-1 L^-1 P^-1 with the
 * triangular inverses taken in fp64 and rounded to fp32 as the reference does (NULL = skip). */
int lfi_invconv_compose(int K, int C, const float *p, const float *l, const float *u, const float *log_s,
                        const float *sign_s, float *w, float *winv, void *ws, size_t ws_bytes, void *stream);
/* chain rule of the composition: dl, du, dlog_s from dW (masked exactly as autograd masks them). */
int lfi_invconv_compose_bwd(int K, int C, const float *p, const float *l, const float *u, const float *log_s,
                            const float *sign_s, const float *dw, float *dl, float *du, float *dlog_s, void *ws,
                            size_t ws_bytes, void *stream);

/* ---- SeqGlow.forward (models.py:534-561): z, per-sample NLL, stash for backward ------------
 * z [T',B,C]; nll [T',B] in bits WITHOUT the parameter-only constant  C*sum_k(sum logs_k + sum log_s_k)
 * (modules.py:62,171), which the host adds (it owns log_s).  scale_out NULL or [K,B,C-C/2]: the
 * last frame's coupling scale per step (FlowStep.scale under scale_logging, models.py:336-337). */
int lfi_seq_train_fwd(const lfi_shape *s, const void *derived, const lfi_params *p, const lfi_batch *b,
                      float *z, float *nll, float *scale_out, void *ws, size_t ws_bytes, int gemm_mode,
                      void *stream);
/* Backward of the above given its output z and dnll [T',B] (dL/dnll); must follow the forward on
 * the same workspace.  Gradients are ACCUMULATED into g (same layout as lfi_params; g->w receives
 * dL/dW of the composed weight). */
int lfi_seq_train_bwd(const lfi_shape *s, const void *derived, const lfi_params *p, const lfi_batch *b,
                      const float *z, const float *dnll, lfi_params *g, void *ws, size_t ws_bytes, int gemm_mode,
                      void *stream);
/* The same backward that also gives dL/d(input streams) (SeqGlow.forward differentiated with respect to its batch, as torch
 * differentiates the reference's per-frame loop).  Arguments as lfi_seq_train_bwd, plus
 *   dx[m]  NULL (not wanted) or [B, T, dim[m]] batch-first: dL/d(b->x[m]), WRITTEN over all T frames.  p1_face gets the gradient
 *          of its windows and of the flow input (frame start_ts + t') as one sum; frames that no window and no flow input reads
 *          are exact zeros.  Dropout masks scale the gradients as they scaled the inputs.  A non-NULL entry for an absent
 *          modality (hist 0) is an argument error.
 *   dws    scratch of lfi_train_dx_ws_bytes bytes (the dXg products of each GRU encoder, whose chains run concurrently).
 * Null required pointers and a too-small ws / dws return a status before anything is launched.  The parameter gradients are
 * those of lfi_seq_train_bwd (same kernels; reduction order may differ in the last bits) and the grad-ready event is recorded at
 * the same point.  Like the parameter gradients of the encoders, the input gradients of GRU modalities are not bit-reproducible
 * (their dh chains accumulate with split-K atomics).  At final_model.yaml, B = 256, T = 80 the scratch is 108.0 MB in every mode (p2_face 77.1, p2_speech 27.5, p1_speech
 * 3.4 MB); with every modality "enc: none" it is the minimal 256 bytes. */
size_t lfi_train_dx_ws_bytes(const lfi_shape *s, int B, int T, int gemm_mode);
int lfi_seq_train_bwd_dx(const lfi_shape *s, const void *derived, const lfi_params *p, const lfi_batch *b,
                         const float *z, const float *dnll, lfi_params *g, void *ws, size_t ws_bytes, float *const dx[LFI_NMOD],
                         void *dws, size_t dws_bytes, int gemm_mode, void *stream);

/* ---- SeqGlow.forward without gradients, in chunks of frames (models.py:534-561 under torch.no_grad()) ---------------------
 * z [T',B,C] and nll [T',B] as lfi_seq_train_fwd (nll without the parameter-only constant, which the host adds); scale_out NULL
 * or [K,B,C-C/2]: the last frame's coupling scale per step.  Dropout masks come in b->mask in the training layout [T',B,hist].
 * The frames are scored `chunk` at a time: per chunk the conditioning, the gate-ih pre-activations, then the forward flow core,
 * which starts from the RNN state the previous chunk left.  Nothing is kept for a backward pass, so the workspace
 * (lfi_eval_ws_bytes) grows with T only by the encoders' per-raw-frame input projections; everything else is sized by the chunk.
 * At final_model.yaml, B = 256 and 56 frames per chunk it is about 2.4 GB in bf16x3, against 11.9 GB for lfi_seq_train_fwd at
 * T = 80.  lfi_eval_ws_bytes returns 0 for a bad shape, chunk < 1 or T <= start_ts.  Null pointers, chunk < 1 or T <= start_ts
 * (LFI_ERR_ARG) and a short workspace (LFI_ERR_WORKSPACE) return a status before anything is launched. */
size_t lfi_eval_ws_bytes(const lfi_shape *s, int B, int T, int chunk, int gemm_mode);
int lfi_seq_eval(const lfi_shape *s, const void *derived, const lfi_params *p, const lfi_batch *b, int chunk, float *z,
                 float *nll, float *scale_out, void *ws, size_t ws_bytes, int gemm_mode, void *stream);

/* ---- SeqGlow.inference (models.py:567-596): persistent autoregressive sampler ---------------
 * faces [B, seq_len, C] in/out: the first start_ts frames hold the seed (data["p1_face"]), frames
 * t >= start_ts are written (prev_p1_faces of models.py:591; the reference returns [:, start_ts:]).
 * Other modalities [B, T>=seq_len, d] (time stride b->T).  noise [T',B,C] (already scaled by eps)
 * or NULL for zeros.  Frames are generated in chunks of `chunk`
 * frames (static conditioning for a chunk is computed time-parallel, then one persistent kernel
 * steps the chunk).  teacher_forced=1 implements SeqGlow.invert (models.py:617-645): noise is the
 * given z sequence, conditioning uses batch.x[0] [B,T,C] ground truth; logdet_out [T',B] optional
 * (coupling terms only, the host adds the parameter-only constant). */
int lfi_seq_sample(const lfi_shape *s, const void *derived, const lfi_params *p, const lfi_batch *b,
                   int seq_len, const float *noise, float *faces, float *logdet_out, int teacher_forced,
                   int chunk, void *ws, size_t ws_bytes, int gemm_mode, void *stream);

/* ---- FeatureEncoder.forward (models.py:127-145) for frames t0..t0+Tp-1: cond [Tp*B, Fe] (folded:
 * each GRU-encoded modality contributes its final state once; the reference concatenates it twice). */
size_t lfi_feature_ws_bytes(const lfi_shape *s, int B, int T, int Tp, int gemm_mode);
int lfi_feature_encode(const lfi_shape *s, const lfi_params *p, const lfi_batch *b, int t0, int Tp, float *cond,
                       void *ws, size_t ws_bytes, int gemm_mode, void *stream);

/* ---- FeatureEncoder / ModalityEncoder.forward WITH autograd (models.py:12-145 differentiated by torch) -----------------------
 * lfi_feature_encode_fwd_train computes the same folded cond [Tp*B, Fe] as lfi_feature_encode, with the window-GRU launches of the
 * training step (per-step fused GRU GEMMs with the input projection inside in the tensor-core modes; never the persistent kernel,
 * which keeps no stash), and fills `stash` (lfi_feature_stash_bytes, caller owned, opaque: h of every window step, the gate stash,
 * the masked window inputs).  One stash per call: a per-frame loop that makes T forward calls before one backward keeps T of them.
 * At final_model.yaml, B = 256, Tp = 1 a stash is 53.7 MB in fp32 mode, 66.5 MB in bf16x3 and 60.1 MB in bf16 mode, most of it
 * p2_face (hist 24, E = 256: 31.5 MB in fp32, 39.1 MB in bf16x3); a 56-frame loop keeps all 56 alive until its backward.
 * lfi_feature_encode_bwd is its backward; it must get the stash of the matching forward call and the same batch, masks and mode.
 *   in : dcond [Tp*B, Fe] = dL/d(folded cond) (the caller sums the two copies of a GRU state of the unfolded vector)
 *   out: dx[m] NULL or [B, T, dim[m]]: dL/d(raw stream m) over all T frames, zero where no window reads a frame (GRU and
 *        "enc: none" modalities; dx itself may be NULL); the enc_* fields of g (layout of lfi_params, nothing else is read) are
 *        WRITTEN, not accumulated.
 * Both take a workspace of at least lfi_feature_bwd_ws_bytes bytes.  Numerics: the GEMMs run in gemm_mode.  In
 * fp32 mode the forward equals lfi_feature_encode bitwise (same kernels); in the tensor-core modes lfi_feature_encode runs the
 * persistent window-GRU kernel, so the two agree within the mode's bound only.  The backward has no atomics and no split-K
 * (weight gradients written by one tile each, bias gradients as per-block partials reduced in a fixed order, the adjoint of the
 * window gather one thread per element): the same call twice gives bit-identical gradients in every mode. */
size_t lfi_feature_stash_bytes(const lfi_shape *s, int B, int T, int Tp, int gemm_mode);
size_t lfi_feature_bwd_ws_bytes(const lfi_shape *s, int B, int T, int Tp, int gemm_mode);
int lfi_feature_encode_fwd_train(const lfi_shape *s, const lfi_params *p, const lfi_batch *b, int t0, int Tp, float *cond,
                                 void *stash, size_t stash_bytes, void *ws, size_t ws_bytes, int gemm_mode, void *stream);
int lfi_feature_encode_bwd(const lfi_shape *s, const lfi_params *p, const lfi_batch *b, int t0, int Tp, const float *dcond,
                           float *const dx[LFI_NMOD], lfi_params *g, void *stash, size_t stash_bytes, void *ws, size_t ws_bytes,
                           int gemm_mode, void *stream);

/* ---- single-frame module API (FlowStep.forward models.py:305-373, test_modules.py) ----------
 * One flow step k on one frame: x [B,C], cond [B,F] (raw, unfolded), h (and c) [B,H] in/out
 * (NULL h_in = zeros, f_seq.init_rnn_hidden), logdet [B] in/out (coupling term only). */
int lfi_flowstep(const lfi_shape *s, const void *derived, const lfi_params *p, int k, int reverse,
                 const float *x, const float *cond, const float *h_in, const float *c_in, float *h_out,
                 float *c_out, float *y, float *logdet, float *scale_out, int B, void *ws, size_t ws_bytes,
                 void *stream);
size_t lfi_flowstep_ws_bytes(const lfi_shape *s, int B);

/* ---- FlowStep.forward WITH autograd (models.py:305-342 under torch autograd; test_modules.py:30-67 builds training loops on
 * the per-frame module API).  lfi_flowstep_fwd_train = lfi_flowstep (forward direction) that also fills `stash`
 * (lfi_flowstep_stash_bytes, caller owned, opaque) with the activations of the call; lfi_flowstep_bwd is its backward:
 *   in : dy [B,C] = dL/d(output), dlogdet [B] = dL/d(logdet) (NULL = 0), dh_out / dc_out [B,H] = dL/d(new state) (NULL = 0),
 *        cond [B,F] and h_in / c_in [B,H] as passed to the forward (NULL state = zeros)
 *   out: dx [B,C], dcond [B,F], dh_in (/ dc_in) [B,H]; parameter gradients of step k are ACCUMULATED into g (layout of
 *        lfi_params; g->w receives dL/dW of the composed 1x1 weight -> lfi_invconv_compose_bwd; the parameter-only log-det
 *        terms C*sum(logs), C*sum(log_s) are the host's, as in lfi_seq_train_bwd). */
size_t lfi_flowstep_stash_bytes(const lfi_shape *s, int B);
size_t lfi_flowstep_bwd_ws_bytes(const lfi_shape *s, int B);
int lfi_flowstep_fwd_train(const lfi_shape *s, const void *derived, const lfi_params *p, int k, const float *x, const float *cond,
                           const float *h_in, const float *c_in, float *h_out, float *c_out, float *y, float *logdet,
                           float *scale_out, int B, void *stash, size_t stash_bytes, void *ws, size_t ws_bytes, void *stream);
int lfi_flowstep_bwd(const lfi_shape *s, const void *derived, const lfi_params *p, int k, const float *cond, const float *h_in,
                     const float *c_in, const float *dy, const float *dlogdet, const float *dh_out, const float *dc_out, float *dx,
                     float *dcond, float *dh_in, float *dc_in, lfi_params *g, int B, void *stash, size_t stash_bytes, void *ws,
                     size_t ws_bytes, void *stream);

/* ---- FlowStep.forward(reverse=True) WITH autograd (FlowStep.reverse_flow models.py:345-373 and FlowNet.decode 444-462 under
 * torch autograd).  lfi_flowstep_rev_fwd_train = lfi_flowstep with reverse=1 (same kernels, bitwise the same outputs) that also
 * fills `stash` (lfi_flowstep_stash_bytes bytes) with the activations of the call; lfi_flowstep_rev_bwd is its backward, with
 * the arguments of lfi_flowstep_bwd (dy = dL/d(output), dx = dL/d(input)) and a workspace of lfi_flowstep_rev_bwd_ws_bytes.
 * Differences from lfi_flowstep_bwd: the parameter gradients of step k are WRITTEN, not accumulated (g->w still receives dL/dW
 * of the composed FORWARD weight, read through W^-1 from the derived cache, which lfi_derive must have built with winv); the
 * reverse log-det subtracts the coupling terms, and the parameter-only terms C*sum(logs), C*sum(log_s) are the host's; every
 * reduction over the B rows runs in a fixed order (no atomics, no split-K), so the same call twice gives bit-identical
 * gradients.  A null pointer, a short stash or a short workspace returns a status before anything is launched. */
size_t lfi_flowstep_rev_bwd_ws_bytes(const lfi_shape *s, int B);
int lfi_flowstep_rev_fwd_train(const lfi_shape *s, const void *derived, const lfi_params *p, int k, const float *x, const float *cond,
                               const float *h_in, const float *c_in, float *h_out, float *c_out, float *y, float *logdet, int B,
                               void *stash, size_t stash_bytes, void *ws, size_t ws_bytes, void *stream);
int lfi_flowstep_rev_bwd(const lfi_shape *s, const void *derived, const lfi_params *p, int k, const float *cond, const float *h_in,
                         const float *c_in, const float *dy, const float *dlogdet, const float *dh_out, const float *dc_out, float *dx,
                         float *dcond, float *dh_in, float *dc_in, lfi_params *g, int B, void *stash, size_t stash_bytes, void *ws,
                         size_t ws_bytes, void *stream);

/* ---- stand-alone modules under autograd (modules.py ActNorm2d / InvertibleConv1x1 / LinearZeros, models.py f_seq) ---------
 * Backward passes of lfi_actnorm and of LinearZeros, and f_seq.forward (models.py:204-214) with its backward, each on the
 * module's own tensors.  GEMMs run in LFI_GEMM_FP32, as in lfi_flowstep.  Parameter gradients are WRITTEN, not accumulated.
 * Every reduction over the B rows runs in a fixed order (no atomics): the same call twice gives bit-identical gradients. */
/* ActNorm2d backward on [B,C]; x / y = input / output of the lfi_actnorm call (reverse=0 reads y, reverse=1 reads x; the
 * other may be NULL).  dbias, dlogs [C]:
 *   reverse=0:  dx = dy e^{logs},   dbias =  sum_B dy e^{logs},  dlogs =  sum_B dy y
 *   reverse=1:  dx = dy e^{-logs},  dbias = -sum_B dy,           dlogs = -sum_B dy x e^{-logs}
 * The parameter-only log-det term C * sum(logs) is the caller's. */
int lfi_actnorm_bwd(const float *x, const float *y, const float *logs, const float *dy, float *dx, float *dbias, float *dlogs,
                    int B, int C, int reverse, void *stream);
/* LinearZeros backward (modules.py:93-95): out = (h W^T + b) e^{f logs}, h [B,In], W [Out,In], f = logscale_factor.  Given
 * out and dout [B,Out]: dh [B,In] = g W, dW [Out,In] = g^T h, db [Out] = sum_B g, dlogs [Out] = f sum_B dout out, with
 * g = dout e^{f logs} (workspace: lfi_linear_zeros_bwd_ws_bytes). */
size_t lfi_linear_zeros_bwd_ws_bytes(int B, int Out);
int lfi_linear_zeros_bwd(const float *h, const float *w, const float *logs, const float *out, const float *dout, float logscale_factor,
                         float *dh, float *dw, float *db, float *dlogs, int B, int In, int Out, void *ws, size_t ws_bytes,
                         void *stream);

/* Shapes of one stand-alone f_seq (models.py:148-194). */
typedef struct lfi_fseq_shape {
  int32_t In;             /* input_size: width of z                                   */
  int32_t Out;            /* output_size: LinearZeros output                          */
  int32_t H;              /* hidden_size                                              */
  int32_t D;              /* cond_dim: cond_transform output                          */
  int32_t F;              /* feature_encoder_dim: width of the conditioning           */
  int32_t G;              /* 3 = GRUCell (r,z,n), 4 = LSTMCell (i,f,g,o)               */
  float logscale_factor;  /* final_linear.logscale_factor (3 by default)              */
} lfi_fseq_shape;

/* Parameters of one f_seq, as the module holds them (not the [K, ...] blocks of lfi_params). */
typedef struct lfi_fseq_params {
  float *wc, *bc;         /* [D,F],[D]         cond_transform.0.{weight,bias}  */
  float *w_ih, *b_ih;     /* [G*H,In+D],[G*H]  rnn.{weight_ih,bias_ih}         */
  float *w_hh, *b_hh;     /* [G*H,H],[G*H]     rnn.{weight_hh,bias_hh}         */
  float *wf, *bf, *lf;    /* [Out,H],[Out],[Out] final_linear.{weight,bias,logs} */
} lfi_fseq_params;

/* f_seq.forward: out [B,Out] = LinearZeros(cell([z | LeakyReLU(cond W_c^T + b_c)], state)), z [B,In], cond [B,F];
 * h_in (c_in) [B,H] or NULL = zeros (f_seq.init_rnn_hidden; the LSTM zero state of FlowStep), h_out (c_out) [B,H].
 * stash NULL (inference) or lfi_fseq_stash_bytes(s, B) bytes, caller owned and opaque, for lfi_fseq_bwd. */
size_t lfi_fseq_ws_bytes(const lfi_fseq_shape *s, int B);
size_t lfi_fseq_stash_bytes(const lfi_fseq_shape *s, int B);
size_t lfi_fseq_bwd_ws_bytes(const lfi_fseq_shape *s, int B);
int lfi_fseq_fwd(const lfi_fseq_shape *s, const lfi_fseq_params *p, const float *z, const float *cond, const float *h_in,
                 const float *c_in, float *h_out, float *c_out, float *out, int B, void *stash, size_t stash_bytes, void *ws,
                 size_t ws_bytes, void *stream);
/* Backward of the above: dout [B,Out], dh_out / dc_out [B,H] = dL/d(new state) (NULL = 0); z, cond, h_in, c_in as passed to
 * the forward.  dz [B,In], dcond [B,F], dh_in / dc_in [B,H] (each NULL = not wanted); all nine parameter gradients are
 * written into g (dW_hh = 0 when h_in is NULL). */
int lfi_fseq_bwd(const lfi_fseq_shape *s, const lfi_fseq_params *p, const float *z, const float *cond, const float *h_in,
                 const float *c_in, const float *dout, const float *dh_out, const float *dc_out, float *dz, float *dcond,
                 float *dh_in, float *dc_in, lfi_fseq_params *g, int B, const void *stash, size_t stash_bytes, void *ws,
                 size_t ws_bytes, void *stream);

/* ---- primitives exposed for the module API and unit parity --------------------------------- */
/* ActNorm2d.forward (modules.py:45-80) on [B,C]: reverse=0  y=(x+bias)*exp(logs); reverse=1 y=x*exp(-logs)-bias */
int lfi_actnorm(const float *x, const float *bias, const float *logs, float *y, int B, int C, int reverse,
                void *stream);
/* C[M,N] = A[M,K] @ B[K,N] (+bias[N]) fp32 — InvertibleConv1x1.forward z = x @ W (modules.py:186) etc. */
int lfi_matmul(const float *a, const float *b, const float *bias, float *c, int M, int N, int K, int transB,
               void *stream);
/* GaussianDiag.logp_simplified + SeqGlow.loss (modules.py:207-212, models.py:563-565):
 * nll[b] = -(logdet[b] + sum_c -0.5 (z^2 + ln 2pi)) / ln 2 */
int lfi_nll(const float *z, const float *logdet, float *nll, int B, int C, void *stream);

/* Output side of sampling (SURVEY.md section 8(f) rank 3): de-standardise the generated frames and scatter the C = exp + jaw +
 * neck channels into the 106-wide FLAME vector the render server consumes - generate_motion_from_model.py:39-51 (expand_face_dim)
 * and :68 (predicted_seq * face_stds + face_means).  x [rows, C] -> out [rows, 106]: out[:, 0:exp] = expression,
 * out[:, 100:100+jaw] = jaw, out[:, 103:103+neck] = neck, every other column 0.  means / stds [C] or NULL (no
 * de-standardisation, the bare expand_face_dim).  The product and the sum are rounded separately, as torch does. */
int lfi_expand_faces(const float *x, const float *means, const float *stds, size_t rows, int exp_dim, int jaw_dim, int neck_dim,
                     float *out, void *stream);

/* Input side on the device (SURVEY.md section 8(f) rank 4): MimicryDataset.__getitem__ + DataLoader collate
 * (mimicry_data_module.py:44-78) over a corpus that stays resident in HBM.  raw [rows, dim]: all segments of one modality back to
 * back; row0 [B] (device, int64): first row of each window (segment offset + window start); out [B, T, dim].  Bit-exact copy. */
int lfi_gather_batch(const float *raw, const long long *row0, int B, int T, int dim, float *out, void *stream);

/* Validation metric on the device (SURVEY.md section 8(f) rank 4): calc_jerk of glow/utils.py:53-58 (mimicry_logger.py:175-184),
 * the mean absolute third difference along time of x [B, T, C] (T >= 4).  scratch8: 8 bytes, 8-byte aligned; out: one float.
 * Differences are three rounded fp32 subtractions as in torch; the mean is accumulated in fp64. */
int lfi_jerk(const float *x, int B, int T, int C, void *scratch8, float *out, void *stream);

/* fused gradient-norm clip + Adam over the flat parameter buffer (lets_face_it_glow.py:61-72,
 * final_model.yaml:126,130): two launches, no host sync.  norm_scratch: 2 floats. */
int lfi_clip_adam(float *theta, float *grad, float *m, float *v, size_t n, float lr, float beta1, float beta2,
                  float eps, float max_norm, float grad_scale, int step, float *norm_scratch, void *stream);

/* The same update with the per-step scalars on the device: hyper[0] = learning rate, hyper[1] = 1 - beta1^step,
 * hyper[2] = sqrt(1 - beta2^step) (computed by the caller in double, as torch.optim.Adam does).  Nothing in the launch
 * arguments changes from step to step, so a whole training step can be captured in a CUDA graph and replayed
 * (SURVEY.md section 8(f) rank 2: graph-capturable optimizer step; train.py: GraphedStep). */
int lfi_clip_adam_dev(float *theta, float *grad, float *m, float *v, size_t n, const float *hyper, float beta1, float beta2,
                      float eps, float max_norm, float grad_scale, float *norm_scratch, void *stream);

/* The same clip followed by torch.optim.SGD or torch.optim.RMSprop (single-tensor semantics of torch 2.x), each as two
 * launches over the flat buffer (the norm pass, then the update) with the per-step scalars read from device memory, so that
 * eager and captured steps run the same launch.  After the clip (g = grad * grad_scale * coef, as lfi_clip_adam):
 *   SGD      g += weight_decay * theta;  with momentum != 0: buf = g on the first momentum step, else
 *            buf = momentum * buf + (1 - dampening) * g, and g = g + momentum * buf (nesterov) or g = buf;  theta -= lr * g
 *   RMSprop  g += weight_decay * theta;  sq = alpha * sq + (1 - alpha) * g^2;  centered (grad_avg given): grad_avg moves
 *            towards g with weight 1 - alpha (torch's lerp_) and avg = sqrt(sq - grad_avg^2) + eps, else avg = sqrt(sq) + eps;
 *            with momentum > 0: buf = momentum * buf + g / avg, theta -= lr * buf, else theta -= lr * g / avg
 * lfi_clip_sgd_dev:     hyper[0] = learning rate, hyper[1] = 1 on the first momentum step (buf holds no value yet and is
 *                       written without being read), else 0.  buf [n] is given exactly when momentum != 0.
 * lfi_clip_rmsprop_dev: hyper[0] = learning rate.  square_avg [n] always; grad_avg [n] or NULL (not centered); buf [n] is
 *                       given exactly when momentum > 0.
 * Bad arguments return LFI_ERR_ARG before anything is launched: a null required pointer, n == 0, a buffer missing for (or
 * given without) the configuration that uses it, a negative momentum / weight_decay (/ alpha / eps), and nesterov without
 * momentum > 0 or with dampening != 0 (torch refuses these too).  The update has no atomics: given the same gradient and
 * norm it is bitwise reproducible.  norm_scratch: 2 floats, as lfi_clip_adam. */
int lfi_clip_sgd_dev(float *theta, float *grad, float *buf, size_t n, const float *hyper, float momentum, float dampening,
                     float weight_decay, int nesterov, float max_norm, float grad_scale, float *norm_scratch, void *stream);
int lfi_clip_rmsprop_dev(float *theta, float *grad, float *square_avg, float *grad_avg, float *buf, size_t n, const float *hyper,
                         float alpha, float eps, float weight_decay, float momentum, float max_norm, float grad_scale,
                         float *norm_scratch, void *stream);

/* generic batched GEMM used by the time-parallel phases (exposed for unit parity of the tcgen05 path)
 * C[b] = op(A[b]) op(B[b]) : transA: A stored [K,M]; transB: B stored [N,K]. epilogue flags below. */
#define LFI_EPI_BIAS 1
#define LFI_EPI_LRELU 2
#define LFI_EPI_ACCUM 4
#define LFI_EPI_LRELU_BWD 8
#define LFI_EPI_ACCUM_PRE 16 /* add the old C before bias/activation: C = act(C + A B + bias) */
int lfi_gemm(int mode, int transA, int transB, int M, int N, int K, const float *A, int lda, long strideA,
             const float *B, int ldb, long strideB, float *C, int ldc, long strideC, const float *bias,
             long strideBias, const float *aux, int ldaux, long strideAux, int batch, int epi, void *ws,
             size_t ws_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* LFI_B200_H */
