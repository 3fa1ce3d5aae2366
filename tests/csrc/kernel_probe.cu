// Test-only entry points into the internals of liblfi_b200.so (tests/test_gpu_kernel_units.py).
//
// The production C ABI (include/lfi_b200.h) reaches the tcgen05 GEMM only through lfi_gemm: fp32 operands and the generic
// epilogues.  The training step and the sampler also use operand planes, plane outputs, the sign-of-plane LeakyReLU', fused
// column sums, the row-interleaved output, the fused encoder-GRU epilogues and the encoder aux kernels.  This library
// exports thin extern "C" wrappers around those internal functions so that the tests can drive them directly.
//
// It defines no kernels and links against the shipped liblfi_b200.so, so the tests check the exact binary the package
// loads.  Argument structs are passed by pointer; tests/kernel_probe.py mirrors them in ctypes, and lfi_probe_layout()
// reports sizeof / offsetof so that a CPU test can compare the mirror with the compiler's layout.
#include <cstddef>
#include <cstring>

#include "../../lets_face_it_b200/csrc/aux_kernels.cuh"
#include "../../lets_face_it_b200/csrc/enc_persist.cuh"
#include "../../lets_face_it_b200/csrc/lfi_common.cuh"

namespace lfi {
size_t gemm_ws_bytes(int mode, const GemmArgs &g);  // gemm_dispatch.cu
}

using lfi::GemmArgs;
using lfi::GruEpi;
using lfi::PlaneRef;
using lfi::aux::EncStep;
using lfi::aux::EncStepBwd2;
using lfi::encp::FwdArgs;

namespace {
struct Field { const char *type, *field; size_t value; };
#define LFI_SZ(T) {#T, "", sizeof(T)}
#define LFI_OFF(T, f) {#T, #f, offsetof(T, f)}
const Field kLayout[] = {
    LFI_SZ(PlaneRef), LFI_OFF(PlaneRef, hi), LFI_OFF(PlaneRef, lo), LFI_OFF(PlaneRef, ld), LFI_OFF(PlaneRef, stride),
    LFI_SZ(GruEpi), LFI_OFF(GruEpi, E), LFI_OFF(GruEpi, s), LFI_OFF(GruEpi, hist), LFI_OFF(GruEpi, B), LFI_OFF(GruEpi, T),
    LFI_OFF(GruEpi, t0), LFI_OFF(GruEpi, gates16), LFI_OFF(GruEpi, xp), LFI_OFF(GruEpi, b_ih), LFI_OFF(GruEpi, b_hh),
    LFI_OFF(GruEpi, mask), LFI_OFF(GruEpi, hprev), LFI_OFF(GruEpi, h), LFI_OFF(GruEpi, gates), LFI_OFF(GruEpi, ahn),
    LFI_OFF(GruEpi, cond), LFI_OFF(GruEpi, cond_ld), LFI_OFF(GruEpi, h_hi), LFI_OFF(GruEpi, h_lo), LFI_OFF(GruEpi, xa_hi),
    LFI_OFF(GruEpi, xa_lo), LFI_OFF(GruEpi, xb_hi), LFI_OFF(GruEpi, xb_lo), LFI_OFF(GruEpi, xa_ld), LFI_OFF(GruEpi, xb_ld),
    LFI_OFF(GruEpi, xk), LFI_OFF(GruEpi, x_only),
    LFI_SZ(GemmArgs), LFI_OFF(GemmArgs, transA), LFI_OFF(GemmArgs, transB), LFI_OFF(GemmArgs, M), LFI_OFF(GemmArgs, N),
    LFI_OFF(GemmArgs, K), LFI_OFF(GemmArgs, A), LFI_OFF(GemmArgs, lda), LFI_OFF(GemmArgs, sA), LFI_OFF(GemmArgs, B),
    LFI_OFF(GemmArgs, ldb), LFI_OFF(GemmArgs, sB), LFI_OFF(GemmArgs, C), LFI_OFF(GemmArgs, ldc), LFI_OFF(GemmArgs, sC),
    LFI_OFF(GemmArgs, bias), LFI_OFF(GemmArgs, sBias), LFI_OFF(GemmArgs, aux), LFI_OFF(GemmArgs, ldaux), LFI_OFF(GemmArgs, sAux),
    LFI_OFF(GemmArgs, batch), LFI_OFF(GemmArgs, epi), LFI_OFF(GemmArgs, pA), LFI_OFF(GemmArgs, pB), LFI_OFF(GemmArgs, pOut),
    LFI_OFF(GemmArgs, fuse), LFI_OFF(GemmArgs, gru), LFI_OFF(GemmArgs, auxp), LFI_OFF(GemmArgs, ldauxp), LFI_OFF(GemmArgs, sAuxp),
    LFI_OFF(GemmArgs, colsum), LFI_OFF(GemmArgs, sColsum), LFI_OFF(GemmArgs, c_tiled32),
    LFI_SZ(EncStep), LFI_OFF(EncStep, xp), LFI_OFF(EncStep, gh), LFI_OFF(EncStep, b_ih), LFI_OFF(EncStep, b_hh), LFI_OFF(EncStep, mask),
    LFI_OFF(EncStep, hprev), LFI_OFF(EncStep, h), LFI_OFF(EncStep, gates), LFI_OFF(EncStep, ahn), LFI_OFF(EncStep, cond),
    LFI_OFF(EncStep, cond_ld), LFI_OFF(EncStep, h_hi), LFI_OFF(EncStep, h_lo), LFI_OFF(EncStep, s), LFI_OFF(EncStep, hist),
    LFI_OFF(EncStep, B), LFI_OFF(EncStep, T), LFI_OFF(EncStep, Tp), LFI_OFF(EncStep, t0), LFI_OFF(EncStep, E), LFI_OFF(EncStep, gates16),
    LFI_SZ(EncStepBwd2), LFI_OFF(EncStepBwd2, gates), LFI_OFF(EncStepBwd2, ahn), LFI_OFF(EncStepBwd2, hprev), LFI_OFF(EncStepBwd2, dh),
    LFI_OFF(EncStepBwd2, dh_extra), LFI_OFF(EncStepBwd2, dh_extra_ld), LFI_OFF(EncStepBwd2, dah32), LFI_OFF(EncStepBwd2, dan32),
    LFI_OFF(EncStepBwd2, dah_hi), LFI_OFF(EncStepBwd2, dah_lo), LFI_OFF(EncStepBwd2, dan_hi), LFI_OFF(EncStepBwd2, dan_lo),
    LFI_OFF(EncStepBwd2, gb_ih), LFI_OFF(EncStepBwd2, gb_hh), LFI_OFF(EncStepBwd2, M), LFI_OFF(EncStepBwd2, E),
    LFI_OFF(EncStepBwd2, gates16),
    LFI_SZ(FwdArgs), LFI_OFF(FwdArgs, E), LFI_OFF(FwdArgs, hist), LFI_OFF(FwdArgs, B), LFI_OFF(FwdArgs, T), LFI_OFF(FwdArgs, t0),
    LFI_OFF(FwdArgs, M), LFI_OFF(FwdArgs, nplanes), LFI_OFF(FwdArgs, xp), LFI_OFF(FwdArgs, b_ih), LFI_OFF(FwdArgs, b_hh),
    LFI_OFF(FwdArgs, mask), LFI_OFF(FwdArgs, whh_hi), LFI_OFF(FwdArgs, whh_lo), LFI_OFF(FwdArgs, cond), LFI_OFF(FwdArgs, cond_ld),
    LFI_OFF(FwdArgs, timing),
};
#undef LFI_SZ
#undef LFI_OFF
}  // namespace

extern "C" {

// sizeof(type) for field == "", offsetof(type, field) otherwise; (size_t)-1 for a name the table does not know
size_t lfi_probe_layout(const char *type, const char *field) {
  for (const Field &f : kLayout)
    if (!strcmp(f.type, type) && !strcmp(f.field, field ? field : "")) return f.value;
  return (size_t)-1;
}

int lfi_probe_gemm(int mode, const GemmArgs *g, void *ws, size_t ws_bytes, void *stream) {
  return lfi::gemm_dispatch(mode, *g, ws, ws_bytes, (cudaStream_t)stream);
}

size_t lfi_probe_gemm_ws_bytes(int mode, const GemmArgs *g) { return lfi::gemm_ws_bytes(mode, *g); }

int lfi_probe_split_to_planes(const float *src, int rows, int cols, int ld, long stride, int batch, void *hi, void *lo, void *stream) {
  return lfi::split_to_planes(src, rows, cols, ld, stride, batch, hi, lo, (cudaStream_t)stream);
}

int lfi_probe_enc_gate_fwd(const EncStep *a, void *stream) { return lfi::aux::enc_gate_fwd(*a, (cudaStream_t)stream); }

int lfi_probe_enc_gate_bwd2(const EncStepBwd2 *a, void *stream) { return lfi::aux::enc_gate_bwd2(*a, (cudaStream_t)stream); }

int lfi_probe_colsum_planes(float *out1, float *out2, int period, int lim2, long so, const void *hi, const void *lo, int ld, long sb,
                            int batch, int rows, int col0, int cols, void *stream) {
  return lfi::aux::colsum_planes(out1, out2, period, lim2, so, hi, lo, ld, sb, batch, rows, col0, cols, (cudaStream_t)stream);
}

int lfi_probe_gather_windows_planes(void *hi, void *lo, int ldp, const float *x, const float *mask, int B, int T, int dim, int hist,
                                    int off, int t0, int Tp, void *stream) {
  return lfi::aux::gather_windows_planes(hi, lo, ldp, x, mask, B, T, dim, hist, off, t0, Tp, (cudaStream_t)stream);
}

int lfi_probe_enc_fwd_supported(int E, int hist, size_t M, int mode) { return lfi::encp::fwd_supported(E, hist, M, mode) ? 1 : 0; }

int lfi_probe_enc_launch_fwd(const FwdArgs *a, void *stream) { return lfi::encp::launch_fwd(*a, (cudaStream_t)stream); }

}  // extern "C"
