// Shared internals of liblfi_b200.so (sm_100a only).  Not part of the public ABI.
#pragma once
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../include/lfi_b200.h"

namespace lfi {

void set_error(const char *fmt, ...);
void count_launches(long n);  // bookkeeping for bench.py's gpu_launches claim

#define LFI_CUDA(call)                                                                        \
  do {                                                                                        \
    cudaError_t e__ = (call);                                                                 \
    if (e__ != cudaSuccess) {                                                                 \
      ::lfi::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      return LFI_ERR_CUDA;                                                                    \
    }                                                                                         \
  } while (0)

#define LFI_LAUNCH_CHECK_N(n)                                                                  \
  do {                                                                                        \
    ::lfi::count_launches(n);                                                                 \
    cudaError_t e__ = cudaGetLastError();                                                     \
    if (e__ != cudaSuccess) {                                                                 \
      ::lfi::set_error("%s:%d: launch -> %s", __FILE__, __LINE__, cudaGetErrorString(e__));    \
      return LFI_ERR_CUDA;                                                                    \
    }                                                                                         \
  } while (0)

#define LFI_LAUNCH_CHECK() LFI_LAUNCH_CHECK_N(1)

#define LFI_TRY(expr)          \
  do {                         \
    int r__ = (expr);          \
    if (r__ != LFI_OK) return r__; \
  } while (0)

#define LFI_REQUIRE(cond, code, ...)  \
  do {                                \
    if (!(cond)) {                    \
      ::lfi::set_error(__VA_ARGS__);  \
      return (code);                  \
    }                                 \
  } while (0)

constexpr float kLn2 = 0.6931471805599453f;
constexpr float kLog2Pi = 1.8378770664093453f;
constexpr float kLeaky = 0.01f;  // nn.LeakyReLU() default slope, models.py:189

__host__ __device__ inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
__host__ __device__ inline size_t round_up_sz(size_t x, size_t m) { return (x + m - 1) / m * m; }

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }
// MUFU-based variants for the fused hot loops (ex2.approx + rcp.approx: ~1e-6 relative, far inside the 1e-4 parity bound)
__device__ __forceinline__ float fast_sigmoid(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float fast_tanh(float x) { return 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * x)); }

inline bool env_flag(const char *name, bool dflt) {
  const char *e = getenv(name);
  return e ? (e[0] != '0') : dflt;
}

// ---- derived shape facts -----------------------------------------------------------------------
struct Dims {
  int C, K, H, D, G, GH, Ci, Cz, Co, affine;
  int Cp, Cop, Cip, Dp;  // row pitches (multiples of 4 floats) of the transposed weight copies
  int F, Fe, Far, start_ts;
  int enc_off[LFI_NMOD];   // column offset of each modality inside the raw feature vector (F)
  int enc_offe[LFI_NMOD];  // column offset inside the folded feature vector (Fe)
  int enc_w[LFI_NMOD];     // raw width, folded width
  int enc_we[LFI_NMOD];
  float eps;
};

inline int make_dims(const lfi_shape *s, Dims *d) {
  LFI_REQUIRE(s && d, LFI_ERR_ARG, "null shape");
  LFI_REQUIRE(s->C >= 2 && s->C <= 256, LFI_ERR_SHAPE, "C=%d out of range [2,256]", s->C);
  LFI_REQUIRE(s->K >= 1 && s->K <= 64, LFI_ERR_SHAPE, "K=%d out of range [1,64]", s->K);
  LFI_REQUIRE(s->H >= 4 && s->H <= 512 && s->H % 4 == 0, LFI_ERR_SHAPE, "H=%d must be a multiple of 4 in [4,512]", s->H);
  LFI_REQUIRE(s->D >= 4 && s->D % 4 == 0 && s->D <= 2048, LFI_ERR_SHAPE, "cond_dim=%d must be a multiple of 4 in [4,2048]", s->D);
  LFI_REQUIRE(s->G == 3 || s->G == 4, LFI_ERR_SHAPE, "G=%d must be 3 (GRU) or 4 (LSTM)", s->G);
  LFI_REQUIRE(s->f_raw > 0 || s->hist[0] >= 1, LFI_ERR_SHAPE, "p1_face history must be >= 1");
  d->C = s->C; d->K = s->K; d->H = s->H; d->D = s->D; d->G = s->G; d->GH = s->G * s->H;
  d->Ci = s->C / 2; d->Cz = s->C - s->C / 2; d->affine = s->affine ? 1 : 0;
  d->Co = d->affine ? 2 * d->Cz : d->Cz;
  d->Cp = round_up(d->C, 4); d->Cop = round_up(d->Co, 4); d->Cip = round_up(d->Ci, 4); d->Dp = d->D;
  d->eps = s->scale_eps;
  int F = 0, Fe = 0, st = 0;
  if (s->f_raw > 0) {  // stand-alone flow steps: raw conditioning matrix, no encoders, no AR window
    for (int m = 0; m < LFI_NMOD; ++m) { d->enc_off[m] = 0; d->enc_offe[m] = 0; d->enc_w[m] = 0; d->enc_we[m] = 0; }
    d->F = s->f_raw; d->Fe = s->f_raw; d->Far = 0; d->start_ts = 0;
    return LFI_OK;
  }
  for (int m = 0; m < LFI_NMOD; ++m) {
    d->enc_off[m] = F; d->enc_offe[m] = Fe; d->enc_w[m] = 0; d->enc_we[m] = 0;
    if (s->hist[m] <= 0) continue;
    LFI_REQUIRE(s->dim[m] >= 1, LFI_ERR_SHAPE, "modality %d: dim must be >= 1", m);
    LFI_REQUIRE(s->ehid[m] >= 0, LFI_ERR_SHAPE, "modality %d: encoder hidden must be >= 0", m);
    if (m == 0) LFI_REQUIRE(s->ehid[0] == 0 && s->dim[0] == s->C, LFI_ERR_SHAPE, "p1_face must be 'enc: none' with dim == C");
    if (s->hist[m] > st) st = s->hist[m];
    if (s->ehid[m] > 0) { d->enc_w[m] = 2 * s->ehid[m]; d->enc_we[m] = s->ehid[m]; }
    else { d->enc_w[m] = s->hist[m] * s->dim[m]; d->enc_we[m] = d->enc_w[m]; }
    F += d->enc_w[m]; Fe += d->enc_we[m];
  }
  d->F = F; d->Fe = Fe; d->Far = s->hist[0] * s->C; d->start_ts = st;
  return LFI_OK;
}

// ---- bump allocator over a caller-provided workspace (dry run when base == nullptr) ------------
struct Bump {
  char *base; size_t off; size_t cap;
  Bump(void *b, size_t c) : base((char *)b), off(0), cap(c) {}
  template <class T> T *take(size_t n) {
    off = round_up_sz(off, 256);
    T *p = base ? (T *)(base + off) : nullptr;
    off += n * sizeof(T);
    return p;
  }
  bool ok() const { return base == nullptr || off <= cap; }
};

// ---- module API: activations of one FlowStep.forward call on [B] rows (caller-owned, opaque, lfi_flowstep_stash_bytes) ----
// Forward direction (lfi_flowstep_fwd_train): y = ActNorm output, zf = 1x1 conv output.  Reverse direction
// (lfi_flowstep_rev_fwd_train): y = x1 = zc W^-1 (input of the reverse ActNorm), zf = zc (coupling output).  Both: Cact = the
// cond_transform output, h / c = the new state, gates / ahn / o as the flow-core stash (core::Stash).
struct StepStash {
  float *Cact, *y, *zf, *h, *c, *gates, *ahn, *o;
  size_t bytes;
};
inline void plan_step_stash(const Dims &d, int B, void *base, StepStash *s) {
  Bump b(base, 0);
  s->Cact = b.take<float>((size_t)B * d.D);
  s->y = b.take<float>((size_t)B * d.C);
  s->zf = b.take<float>((size_t)B * d.C);
  s->h = b.take<float>((size_t)B * d.H);
  s->c = b.take<float>((size_t)B * d.H);
  s->gates = b.take<float>((size_t)B * d.GH);
  s->ahn = b.take<float>((size_t)B * d.H);
  s->o = b.take<float>((size_t)B * d.Co);
  s->bytes = round_up_sz(b.off, 256);
}

// ---- generic GEMM (gemm_simt.cu / gemm_tc.cu) ---------------------------------------------------
// bf16 operand planes of the tensor-core modes: value = hi (+ lo in the split-bf16 x3 mode); layout as the fp32
// operand they stand for (same rows / cols / transposition), pitch ld in elements (multiple of 8), 16-byte aligned.
struct PlaneRef {
  const void *hi, *lo;
  int ld; long stride;
};

// Fused encoder-GRU epilogues of the tcgen05 GEMM (ModalityEncoder nn.GRU, models.py:21-27, 63-64): the window step's
// recurrent product h_{s-1} W_hh^T leaves TMEM straight into the gate math, so the [M, 3E] pre-activation matrix never
// travels through HBM.  Argument meaning as aux::EncStep.
// LFI_FUSE_GRU_FWD_X: as _FWD, and the input projection of the step joins the same accumulator: the masked window inputs of
// step s (operand planes [M, xk], as gathered for the dW_ih GEMMs) times W_ih^T run as extra k-blocks - r and u on top of the
// recurrent product, the n gate's input part into a fourth column group (it stays outside r * (...)) - so the epilogue has no
// [M, 3E] projection rows to fetch (three of its four 16-byte load streams).
enum { LFI_FUSE_NONE = 0, LFI_FUSE_GRU_FWD = 1, LFI_FUSE_GRU_FWD_X = 3 };
// 16-bit fixed-point gate stash of the encoder GRUs (tensor-core modes): r, u in [0,1] as unorm16 (|err| <= 7.7e-6), n in
// [-1,1] as snorm16 (|err| <= 1.6e-5).  The forward pass itself uses the exact fp32 gates; only the backward pass reads
// the stash, and its gradient tolerance (5e-3 relative L2 per tensor in bf16x3 mode) is ~100x above the induced error.
__device__ __forceinline__ unsigned short q_unorm16(float v) { return (unsigned short)__float2uint_rn(fminf(fmaxf(v, 0.f), 1.f) * 65535.0f); }
__device__ __forceinline__ unsigned short q_snorm16(float v) { return (unsigned short)(short)__float2int_rn(fminf(fmaxf(v, -1.f), 1.f) * 32767.0f); }
__device__ __forceinline__ float dq_unorm16(unsigned short q) { return (float)q * (1.0f / 65535.0f); }
__device__ __forceinline__ float dq_snorm16(unsigned short q) { return (float)(short)q * (1.0f / 32767.0f); }

struct GruEpi {
  int E, s, hist, B, T, t0;
  int gates16;  // gates stash in 16-bit fixed point ([M][3E] unsigned short in the same buffer)
  // forward (step s >= 1)
  const float *xp, *b_ih, *b_hh, *mask, *hprev;
  float *h, *gates, *ahn, *cond; int cond_ld;
  void *h_hi, *h_lo;
  // LFI_FUSE_GRU_FWD_X: masked window inputs of this step [M, xk] and W_ih [3E, xk] as operand planes (pitches in elements)
  const void *xa_hi, *xa_lo, *xb_hi, *xb_lo; int xa_ld, xb_ld, xk;
  int x_only;  // window step 0: zero state, no recurrent product - the launch consists of the input part alone (hprev == nullptr)
};

struct GemmArgs {
  int transA, transB, M, N, K;
  const float *A; int lda; long sA;
  const float *B; int ldb; long sB;
  float *C; int ldc; long sC;
  const float *bias; long sBias;
  const float *aux; int ldaux; long sAux;
  int batch, epi;
  PlaneRef pA, pB;  // hi != nullptr: operand already split (A / B may then be null); tensor-core modes only
  PlaneRef pOut;    // hi != nullptr: also emit the result as bf16 planes (C may then be null); tensor-core modes only
  int fuse;         // LFI_FUSE_*: replaces the generic epilogue (operands must be planes; tensor-core modes only)
  GruEpi gru;
  // tensor-core modes only: LeakyReLU' mask taken from the sign of a bf16 plane (instead of the fp32 `aux`), and column sums
  // of the final values accumulated into colsum[n] (bias gradients without a second pass over the output)
  const void *auxp; int ldauxp; long sAuxp;
  float *colsum; long sColsum;
  // tensor-core modes only: C is written row-interleaved, element (m, n) at ((m/32) * (ldc/4) + n/4) * 128 + (m%32) * 4 + n%4
  // (+ the batch offset sC): 32 consecutive rows of one 4-column group are contiguous, which is what the thread-per-sequence
  // flow-core kernel reads (core_pipe.cuh: g_tiled_off).  No accumulate epilogues.
  int c_tiled32;
};
int gemm_simt(const GemmArgs &g, cudaStream_t st);
int gemm_dispatch(int mode, const GemmArgs &g, void *ws, size_t ws_bytes, cudaStream_t st);
bool gemm_tc_wants(const GemmArgs &g);
int split_to_planes(const float *src, int rows, int cols, int ld, long stride, int batch, void *hi, void *lo, cudaStream_t st);
inline PlaneRef plane_ref(const void *hi, const void *lo, int ld, long stride = 0) { PlaneRef r; r.hi = hi; r.lo = lo; r.ld = ld; r.stride = stride; return r; }

inline GemmArgs gemm_args(int tA, int tB, int M, int N, int K, const float *A, int lda, const float *B, int ldb,
                          float *C, int ldc, int epi = 0, const float *bias = nullptr) {
  GemmArgs g; memset(&g, 0, sizeof(g));
  g.transA = tA; g.transB = tB; g.M = M; g.N = N; g.K = K; g.A = A; g.lda = lda; g.B = B; g.ldb = ldb;
  g.C = C; g.ldc = ldc; g.batch = 1; g.epi = epi; g.bias = bias;
  return g;
}

}  // namespace lfi
