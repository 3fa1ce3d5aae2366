// Small HBM-bound kernels around the GEMMs and the flow core: layout transforms of the derived weight
// cache, window gathers, encoder GRU gate math, column sums, LU parametrisation helpers, clip + Adam.
// All are coalesced, grid-stride where the size warrants it, warp-shuffle reduced.
#include "aux_kernels.cuh"
#include <cmath>
#include <cuda_bf16.h>

namespace lfi {
namespace aux {

namespace {
constexpr int TB = 256;
inline int blocks_for(size_t n, int per = TB, int cap = 148 * 16) {
  size_t b = (n + per - 1) / per;
  if (b < 1) b = 1;
  if (b > (size_t)cap) b = cap;
  return (int)b;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
}  // namespace

// ------------------------------------------------------------------------------------------------
__global__ void gather2d_kernel(float *dst, int ld, const float *src, long sb, long si, long sj, int batch, int rows, int cols) {
  const size_t n = (size_t)batch * rows * ld;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const int j = (int)(e % ld);
    const size_t q = e / ld;
    const int i = (int)(q % rows), b = (int)(q / rows);
    dst[e] = j < cols ? src[(size_t)b * sb + (size_t)i * si + (size_t)j * sj] : 0.f;
  }
}
int gather2d(float *dst, int ld, const float *src, long sb, long si, long sj, int batch, int rows, int cols, cudaStream_t st) {
  gather2d_kernel<<<blocks_for((size_t)batch * rows * ld), TB, 0, st>>>(dst, ld, src, sb, si, sj, batch, rows, cols);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

struct FoldMap { int off[LFI_NMOD], offe[LFI_NMOD], we[LFI_NMOD], dup[LFI_NMOD]; int F, Fe; };
static FoldMap make_fold(const Dims &d, const lfi_shape &s) {
  FoldMap f;
  for (int m = 0; m < LFI_NMOD; ++m) {
    f.off[m] = d.enc_off[m]; f.offe[m] = d.enc_offe[m]; f.we[m] = d.enc_we[m];
    f.dup[m] = (s.f_raw <= 0 && s.hist[m] > 0 && s.ehid[m] > 0) ? 1 : 0;
  }
  f.F = d.F; f.Fe = d.Fe;
  return f;
}
__global__ void fold_wc_kernel(float *wcf, const float *wc, FoldMap f, size_t rows) {
  const size_t n = rows * f.Fe;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const int j = (int)(e % f.Fe);
    const size_t r = e / f.Fe;
    int m = 0;
#pragma unroll
    for (int i = 1; i < LFI_NMOD; ++i) if (f.we[i] > 0 && j >= f.offe[i]) m = i;
    const int jj = j - f.offe[m];
    const float *src = wc + r * f.F + f.off[m] + jj;
    wcf[e] = f.dup[m] ? src[0] + src[f.we[m]] : src[0];
  }
}
int fold_wc(float *wcf, const float *wc, const Dims &d, const lfi_shape &s, cudaStream_t st) {
  const size_t rows = (size_t)d.K * d.D;
  fold_wc_kernel<<<blocks_for(rows * d.Fe), TB, 0, st>>>(wcf, wc, make_fold(d, s), rows);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}
__global__ void unfold_wc_grad_kernel(float *dwc, const float *dwcf, FoldMap f, size_t rows) {
  const size_t n = rows * f.Fe;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const int j = (int)(e % f.Fe);
    const size_t r = e / f.Fe;
    int m = 0;
#pragma unroll
    for (int i = 1; i < LFI_NMOD; ++i) if (f.we[i] > 0 && j >= f.offe[i]) m = i;
    const int jj = j - f.offe[m];
    float *dst = dwc + r * f.F + f.off[m] + jj;
    const float g = dwcf[e];
    dst[0] += g;
    if (f.dup[m]) dst[f.we[m]] += g;
  }
}
int unfold_wc_grad(float *dwc, const float *dwcf, const Dims &d, const lfi_shape &s, cudaStream_t st) {
  const size_t rows = (size_t)d.K * d.D;
  unfold_wc_grad_kernel<<<blocks_for(rows * d.Fe), TB, 0, st>>>(dwc, dwcf, make_fold(d, s), rows);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

// ------------------------------------------------------------------------------------------------
// column sums: block = 32 columns x 8 row lanes, grid.y splits the rows; one atomic per column per block
__global__ void colsum_kernel(float *out, const float *A, int ld, int rows, int cols, float scale, int rows_per_block) {
  __shared__ float part[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + tx;
  const int r0 = blockIdx.y * rows_per_block, r1 = min(rows, r0 + rows_per_block);
  float s = 0.f;
  if (j < cols)
    for (int r = r0 + ty; r < r1; r += 8) s += A[(size_t)r * ld + j];
  part[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && j < cols) {
#pragma unroll
    for (int i = 1; i < 8; ++i) s += part[i][tx];
    atomicAdd(out + j, s * scale);
  }
}
int colsum(float *out, const float *A, int ld, int rows, int cols, float scale, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return LFI_OK;
  const int cb = (cols + 31) / 32;
  int rb = (148 * 8 + cb - 1) / cb;
  const int maxrb = (rows + 63) / 64;
  if (rb > maxrb) rb = maxrb;
  if (rb < 1) rb = 1;
  const int rpb = (rows + rb - 1) / rb;
  colsum_kernel<<<dim3(cb, rb), 256, 0, st>>>(out, A, ld, rows, cols, scale, rpb);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

// ------------------------------------------------------------------------------------------------
__global__ void actnorm_kernel(const float *x, const float *bias, const float *logs, float *y, size_t n, int C, int reverse) {
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % C);
    y[e] = reverse ? x[e] * expf(-logs[c]) - bias[c] : (x[e] + bias[c]) * expf(logs[c]);
  }
}
int actnorm(const float *x, const float *bias, const float *logs, float *y, int B, int C, int reverse, cudaStream_t st) {
  actnorm_kernel<<<blocks_for((size_t)B * C), TB, 0, st>>>(x, bias, logs, y, (size_t)B * C, C, reverse);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

__global__ void nll_kernel(const float *z, const float *logdet, float *out, int B, int C) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= B) return;
  float s = 0.f;
  for (int c = lane; c < C; c += 32) { const float v = z[(size_t)b * C + c]; s += v * v; }
  s = warp_sum(s);
  if (lane == 0) out[b] = -(logdet[b] - 0.5f * (s + (float)C * kLog2Pi)) / kLn2;
}
int nll(const float *z, const float *logdet, float *out, int B, int C, cudaStream_t st) {
  nll_kernel<<<(B + 7) / 8, 256, 0, st>>>(z, logdet, out, B, C);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

// ------------------------------------------------------------------------------------------------
__global__ void gather_windows_kernel(float *dst, int ld, int layout_steps, const float *x, const float *mask, int B, int T,
                                      int dim, int hist, int off, int t0, int Tp) {
  const size_t M = (size_t)Tp * B;
  const size_t n = M * hist * dim;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % dim);
    size_t q = e / dim;
    int s; size_t m;
    if (layout_steps) { m = q % M; s = (int)(q / M); }
    else { s = (int)(q % hist); m = q / hist; }
    const int b = (int)(m % B), tp = (int)(m / B);
    const int tau = t0 + tp - hist + off + s;
    float v = x[((size_t)b * T + tau) * dim + c];
    if (mask) v *= mask[m * hist + s];
    if (layout_steps) dst[((size_t)s * M + m) * ld + c] = v;
    else dst[m * ld + (size_t)s * dim + c] = v;
  }
}
int gather_windows(float *dst, int ld, int layout_steps, const float *x, const float *mask, int B, int T, int dim, int hist,
                   int off, int t0, int Tp, cudaStream_t st) {
  gather_windows_kernel<<<blocks_for((size_t)Tp * B * hist * dim), TB, 0, st>>>(dst, ld, layout_steps, x, mask, B, T, dim,
                                                                                hist, off, t0, Tp);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

// ------------------------------------------------------------------------------------------------
// thread = 8 consecutive input features of one (window step, window): 16-byte stores into each plane
__global__ void gather_windows_planes_kernel(__nv_bfloat16 *__restrict__ hi, __nv_bfloat16 *__restrict__ lo, int ldp, const float *__restrict__ x,
                                             const float *__restrict__ mask, int B, int T, int dim, int hist, int off, int t0, int Tp) {
  const size_t M = (size_t)Tp * B;
  const int groups = ldp >> 3;
  const size_t n = M * hist * groups;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const int c0 = (int)(e % groups) * 8;
    const size_t q = e / groups;
    const size_t m = q % M;
    const int s = (int)(q / M);
    const int b = (int)(m % B), tp = (int)(m / B);
    const int tau = t0 + tp - hist + off + s;
    const float *src = x + ((size_t)b * T + tau) * dim + c0;
    const float mk = mask ? mask[m * hist + s] : 1.0f;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = (c0 + j < dim) ? src[j] * mk : 0.f;
    __align__(16) __nv_bfloat16 h8[8], l8[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      h8[j] = __float2bfloat16_rn(v[j]);
      l8[j] = __float2bfloat16_rn(v[j] - __bfloat162float(h8[j]));
    }
    const size_t o = ((size_t)s * M + m) * ldp + c0;
    *reinterpret_cast<uint4 *>(hi + o) = *reinterpret_cast<const uint4 *>(h8);
    if (lo) *reinterpret_cast<uint4 *>(lo + o) = *reinterpret_cast<const uint4 *>(l8);
  }
}
int gather_windows_planes(void *hi, void *lo, int ldp, const float *x, const float *mask, int B, int T, int dim, int hist, int off, int t0,
                          int Tp, cudaStream_t st) {
  LFI_REQUIRE(ldp % 8 == 0 && ldp >= dim && (((uintptr_t)hi | (uintptr_t)lo) & 15) == 0, LFI_ERR_ARG, "gather_windows_planes: plane pitch / alignment");
  gather_windows_planes_kernel<<<blocks_for((size_t)Tp * B * hist * (ldp / 8)), TB, 0, st>>>((__nv_bfloat16 *)hi, (__nv_bfloat16 *)lo, ldp, x, mask, B,
                                                                                             T, dim, hist, off, t0, Tp);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

// ------------------------------------------------------------------------------------------------
__global__ void enc_gate_fwd_kernel(EncStep a) {
  const size_t M = (size_t)a.Tp * a.B;
  const int E = a.E;
  const size_t n = M * E;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < n; idx += (size_t)gridDim.x * blockDim.x) {
    const int e = (int)(idx % E);
    const size_t m = idx / E;
    const int b = (int)(m % a.B), tp = (int)(m / a.B);
    const int tau = a.t0 + tp - a.hist + 1 + a.s;
    const float mk = a.mask ? a.mask[m * a.hist + a.s] : 1.0f;
    const float *xp = a.xp + ((size_t)b * a.T + tau) * 3 * E;
    const float air = mk * xp[e] + a.b_ih[e], aiu = mk * xp[E + e] + a.b_ih[E + e], ain = mk * xp[2 * E + e] + a.b_ih[2 * E + e];
    float ahr = a.b_hh[e], ahu = a.b_hh[E + e], ahn = a.b_hh[2 * E + e];
    float hp = 0.f;
    if (a.gh) {
      const float *g = a.gh + m * 3 * E;
      ahr += g[e]; ahu += g[E + e]; ahn += g[2 * E + e];
    }
    if (a.hprev) hp = a.hprev[idx];
    const float rg = sigmoidf_(air + ahr), ug = sigmoidf_(aiu + ahu);
    const float ng = tanhf(ain + rg * ahn);
    const float h = ng + ug * (hp - ng);
    a.h[idx] = h;
    if (a.gates && a.gates16) {
      unsigned short *g = reinterpret_cast<unsigned short *>(a.gates) + m * 3 * E;
      g[e] = q_unorm16(rg); g[E + e] = q_unorm16(ug); g[2 * E + e] = q_snorm16(ng);
    } else if (a.gates) { float *g = a.gates + m * 3 * E; g[e] = rg; g[E + e] = ug; g[2 * E + e] = ng; }
    if (a.ahn) a.ahn[idx] = ahn;
    if (a.cond) a.cond[m * a.cond_ld + e] = h;
    if (a.h_hi) {
      const __nv_bfloat16 hh = __float2bfloat16_rn(h);
      ((__nv_bfloat16 *)a.h_hi)[idx] = hh;
      if (a.h_lo) ((__nv_bfloat16 *)a.h_lo)[idx] = __float2bfloat16_rn(h - __bfloat162float(hh));
    }
  }
}
// Vectorised variant (E % 4 == 0, 16-byte aligned streams): thread = 4 consecutive hidden units of one window
__global__ void enc_gate_fwd_v4_kernel(EncStep a) {
  const size_t M = (size_t)a.Tp * a.B;
  const int E = a.E, E4 = E >> 2;
  const size_t n = M * E4;
  for (size_t i4 = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i4 < n; i4 += (size_t)gridDim.x * blockDim.x) {
    const int e = (int)(i4 % E4) * 4;
    const size_t m = i4 / E4;
    const size_t idx = m * E + e;
    const int b = (int)(m % a.B), tp = (int)(m / a.B);
    const int tau = a.t0 + tp - a.hist + 1 + a.s;
    const float mk = a.mask ? a.mask[m * a.hist + a.s] : 1.0f;
    const float *xp = a.xp + ((size_t)b * a.T + tau) * 3 * E + e;
    const float4 xr = *reinterpret_cast<const float4 *>(xp), xu = *reinterpret_cast<const float4 *>(xp + E), xn = *reinterpret_cast<const float4 *>(xp + 2 * E);
    const float4 bir = *reinterpret_cast<const float4 *>(a.b_ih + e), biu = *reinterpret_cast<const float4 *>(a.b_ih + E + e),
                 bin = *reinterpret_cast<const float4 *>(a.b_ih + 2 * E + e);
    float4 ahr = *reinterpret_cast<const float4 *>(a.b_hh + e), ahu = *reinterpret_cast<const float4 *>(a.b_hh + E + e),
           ahn = *reinterpret_cast<const float4 *>(a.b_hh + 2 * E + e);
    if (a.gh) {
      const float *g = a.gh + m * 3 * E + e;
      const float4 gr = *reinterpret_cast<const float4 *>(g), gu = *reinterpret_cast<const float4 *>(g + E), gn = *reinterpret_cast<const float4 *>(g + 2 * E);
      ahr.x += gr.x; ahr.y += gr.y; ahr.z += gr.z; ahr.w += gr.w;
      ahu.x += gu.x; ahu.y += gu.y; ahu.z += gu.z; ahu.w += gu.w;
      ahn.x += gn.x; ahn.y += gn.y; ahn.z += gn.z; ahn.w += gn.w;
    }
    const float4 hp = a.hprev ? *reinterpret_cast<const float4 *>(a.hprev + idx) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float xr_[4] = {xr.x, xr.y, xr.z, xr.w}, xu_[4] = {xu.x, xu.y, xu.z, xu.w}, xn_[4] = {xn.x, xn.y, xn.z, xn.w};
    const float bir_[4] = {bir.x, bir.y, bir.z, bir.w}, biu_[4] = {biu.x, biu.y, biu.z, biu.w}, bin_[4] = {bin.x, bin.y, bin.z, bin.w};
    const float ahr_[4] = {ahr.x, ahr.y, ahr.z, ahr.w}, ahu_[4] = {ahu.x, ahu.y, ahu.z, ahu.w}, ahn_[4] = {ahn.x, ahn.y, ahn.z, ahn.w};
    const float hp_[4] = {hp.x, hp.y, hp.z, hp.w};
    float rg[4], ug[4], ng[4], h[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {  // same arithmetic as the scalar kernel
      rg[c] = sigmoidf_(mk * xr_[c] + bir_[c] + ahr_[c]);
      ug[c] = sigmoidf_(mk * xu_[c] + biu_[c] + ahu_[c]);
      ng[c] = tanhf(mk * xn_[c] + bin_[c] + rg[c] * ahn_[c]);
      h[c] = ng[c] + ug[c] * (hp_[c] - ng[c]);
    }
    *reinterpret_cast<float4 *>(a.h + idx) = make_float4(h[0], h[1], h[2], h[3]);
    if (a.gates && a.gates16) {
      unsigned short *g = reinterpret_cast<unsigned short *>(a.gates) + m * 3 * E + e;
      *reinterpret_cast<uint2 *>(g) = make_uint2(q_unorm16(rg[0]) | ((unsigned)q_unorm16(rg[1]) << 16), q_unorm16(rg[2]) | ((unsigned)q_unorm16(rg[3]) << 16));
      *reinterpret_cast<uint2 *>(g + E) = make_uint2(q_unorm16(ug[0]) | ((unsigned)q_unorm16(ug[1]) << 16), q_unorm16(ug[2]) | ((unsigned)q_unorm16(ug[3]) << 16));
      *reinterpret_cast<uint2 *>(g + 2 * E) = make_uint2(q_snorm16(ng[0]) | ((unsigned)q_snorm16(ng[1]) << 16), q_snorm16(ng[2]) | ((unsigned)q_snorm16(ng[3]) << 16));
    } else if (a.gates) {
      float *g = a.gates + m * 3 * E + e;
      *reinterpret_cast<float4 *>(g) = make_float4(rg[0], rg[1], rg[2], rg[3]);
      *reinterpret_cast<float4 *>(g + E) = make_float4(ug[0], ug[1], ug[2], ug[3]);
      *reinterpret_cast<float4 *>(g + 2 * E) = make_float4(ng[0], ng[1], ng[2], ng[3]);
    }
    if (a.ahn) *reinterpret_cast<float4 *>(a.ahn + idx) = ahn;
    if (a.cond) {
      float *cd = a.cond + m * a.cond_ld + e;
      cd[0] = h[0]; cd[1] = h[1]; cd[2] = h[2]; cd[3] = h[3];
    }
    if (a.h_hi) {
      __align__(8) __nv_bfloat16 h4[4], l4[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) { h4[c] = __float2bfloat16_rn(h[c]); l4[c] = __float2bfloat16_rn(h[c] - __bfloat162float(h4[c])); }
      *reinterpret_cast<uint2 *>((__nv_bfloat16 *)a.h_hi + idx) = *reinterpret_cast<const uint2 *>(h4);
      if (a.h_lo) *reinterpret_cast<uint2 *>((__nv_bfloat16 *)a.h_lo + idx) = *reinterpret_cast<const uint2 *>(l4);
    }
  }
}
int enc_gate_fwd(const EncStep &a, cudaStream_t st) {
  auto al16 = [](const void *p) { return p == nullptr || ((uintptr_t)p & 15) == 0; };
  if (a.E % 4 == 0 && al16(a.xp) && al16(a.gh) && al16(a.b_ih) && al16(a.b_hh) && al16(a.hprev) && al16(a.h) && al16(a.gates) && al16(a.ahn) &&
      (((uintptr_t)a.h_hi | (uintptr_t)a.h_lo) & 7) == 0) {
    enc_gate_fwd_v4_kernel<<<blocks_for((size_t)a.Tp * a.B * (a.E / 4)), TB, 0, st>>>(a);
    LFI_LAUNCH_CHECK();
    return LFI_OK;
  }
  enc_gate_fwd_kernel<<<blocks_for((size_t)a.Tp * a.B * a.E), TB, 0, st>>>(a);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

// thread = hidden unit e (coalesced over e), block = a strip of rows; the four bias-gradient sums stay in registers
// kPart: the block adds its sums into its own row of part [blocks][4E] instead of issuing atomics
template <bool kPart>
__global__ void enc_gate_bwd2_kernel(EncStepBwd2 a, int rows_per_block, float *part) {
  const int E = a.E;
  const int e = blockIdx.y * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const int r0 = blockIdx.x * rows_per_block, r1 = min(a.M, r0 + rows_per_block);
  float s_r = 0.f, s_u = 0.f, s_n = 0.f, s_nr = 0.f;
  __nv_bfloat16 *dah_hi = (__nv_bfloat16 *)a.dah_hi, *dah_lo = (__nv_bfloat16 *)a.dah_lo;
  __nv_bfloat16 *dan_hi = (__nv_bfloat16 *)a.dan_hi, *dan_lo = (__nv_bfloat16 *)a.dan_lo;
  auto put = [](__nv_bfloat16 *hi, __nv_bfloat16 *lo, size_t o, float v) {
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    hi[o] = h;
    if (lo) lo[o] = __float2bfloat16_rn(v - __bfloat162float(h));
  };
  for (int m = r0; m < r1; ++m) {
    const size_t idx = (size_t)m * E + e, g3 = (size_t)m * 3 * E;
    float dh = a.dh[idx];
    if (a.dh_extra) dh += a.dh_extra[(size_t)m * a.dh_extra_ld + e];
    float rg, ug, ng;
    if (a.gates16) {
      const unsigned short *gq = reinterpret_cast<const unsigned short *>(a.gates);
      rg = dq_unorm16(gq[g3 + e]); ug = dq_unorm16(gq[g3 + E + e]); ng = dq_snorm16(gq[g3 + 2 * E + e]);
    } else {
      rg = a.gates[g3 + e]; ug = a.gates[g3 + E + e]; ng = a.gates[g3 + 2 * E + e];
    }
    const float hp = a.hprev ? a.hprev[idx] : 0.f;
    const float an = a.ahn[idx];
    const float dn = dh * (1.0f - ug), du = dh * (hp - ng);
    const float dan = dn * (1.0f - ng * ng), dau = du * ug * (1.0f - ug), dar = dan * an * rg * (1.0f - rg);
    const float danr = dan * rg;
    if (a.dah32) { a.dah32[g3 + e] = dar; a.dah32[g3 + E + e] = dau; a.dah32[g3 + 2 * E + e] = danr; a.dan32[idx] = dan; }
    if (dah_hi) {
      put(dah_hi, dah_lo, g3 + e, dar); put(dah_hi, dah_lo, g3 + E + e, dau); put(dah_hi, dah_lo, g3 + 2 * E + e, danr);
      put(dan_hi, dan_lo, idx, dan);
    }
    a.dh[idx] = dh * ug;
    s_r += dar; s_u += dau; s_n += dan; s_nr += danr;
  }
  if (kPart) {
    float *q = part + (size_t)blockIdx.x * 4 * E + e;
    q[0] += s_r; q[E] += s_u; q[2 * E] += s_n; q[3 * E] += s_nr;
    return;
  }
  atomicAdd(a.gb_ih + e, s_r); atomicAdd(a.gb_ih + E + e, s_u); atomicAdd(a.gb_ih + 2 * E + e, s_n);
  atomicAdd(a.gb_hh + e, s_r); atomicAdd(a.gb_hh + E + e, s_u); atomicAdd(a.gb_hh + 2 * E + e, s_nr);
}
// Vectorised variant (E % 4 == 0, 256 % (E/4) == 0): thread = 4 consecutive hidden units of one window, 128-bit loads,
// 64-bit plane stores, grid-stride over the windows so that every SM keeps several independent rows in flight; the
// bias-gradient sums are reduced over the block's row lanes in shared memory before the atomics (kPart: before the block
// adds them into its own row of part [blocks][4E]).
template <bool kPart>
__global__ void __launch_bounds__(256) enc_gate_bwd2_v4_kernel(EncStepBwd2 a, float *part) {
  extern __shared__ float red[];  // [4 sums][rows per iteration][E]
  const int E = a.E, tpr = E >> 2, rpb = 256 / tpr;
  const int e = 4 * (threadIdx.x % tpr), rl = threadIdx.x / tpr;
  float s_r[4] = {0.f, 0.f, 0.f, 0.f}, s_u[4] = {0.f, 0.f, 0.f, 0.f}, s_n[4] = {0.f, 0.f, 0.f, 0.f}, s_nr[4] = {0.f, 0.f, 0.f, 0.f};
  __nv_bfloat16 *dah_hi = (__nv_bfloat16 *)a.dah_hi, *dah_lo = (__nv_bfloat16 *)a.dah_lo;
  __nv_bfloat16 *dan_hi = (__nv_bfloat16 *)a.dan_hi, *dan_lo = (__nv_bfloat16 *)a.dan_lo;
  auto put4 = [](__nv_bfloat16 *hi, __nv_bfloat16 *lo, size_t o, const float (&v)[4]) {
    __align__(8) __nv_bfloat16 h4[4], l4[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) { h4[c] = __float2bfloat16_rn(v[c]); l4[c] = __float2bfloat16_rn(v[c] - __bfloat162float(h4[c])); }
    *reinterpret_cast<uint2 *>(hi + o) = *reinterpret_cast<const uint2 *>(h4);
    if (lo) *reinterpret_cast<uint2 *>(lo + o) = *reinterpret_cast<const uint2 *>(l4);
  };
  for (int m = blockIdx.x * rpb + rl; m < a.M; m += gridDim.x * rpb) {
    const size_t idx = (size_t)m * E + e, g3 = (size_t)m * 3 * E + e;
    float4 d4 = *reinterpret_cast<const float4 *>(a.dh + idx);
    float4 r4, u4, n4;
    if (a.gates16) {
      const unsigned short *gq = reinterpret_cast<const unsigned short *>(a.gates);
      const uint2 rq = __ldg(reinterpret_cast<const uint2 *>(gq + g3)), uq = __ldg(reinterpret_cast<const uint2 *>(gq + g3 + E)),
                  nq = __ldg(reinterpret_cast<const uint2 *>(gq + g3 + 2 * E));
      r4 = make_float4(dq_unorm16(rq.x & 0xffff), dq_unorm16(rq.x >> 16), dq_unorm16(rq.y & 0xffff), dq_unorm16(rq.y >> 16));
      u4 = make_float4(dq_unorm16(uq.x & 0xffff), dq_unorm16(uq.x >> 16), dq_unorm16(uq.y & 0xffff), dq_unorm16(uq.y >> 16));
      n4 = make_float4(dq_snorm16(nq.x & 0xffff), dq_snorm16(nq.x >> 16), dq_snorm16(nq.y & 0xffff), dq_snorm16(nq.y >> 16));
    } else {
      r4 = __ldg(reinterpret_cast<const float4 *>(a.gates + g3)); u4 = __ldg(reinterpret_cast<const float4 *>(a.gates + g3 + E));
      n4 = __ldg(reinterpret_cast<const float4 *>(a.gates + g3 + 2 * E));
    }
    const float4 a4 = __ldg(reinterpret_cast<const float4 *>(a.ahn + idx));
    const float4 h4 = a.hprev ? __ldg(reinterpret_cast<const float4 *>(a.hprev + idx)) : make_float4(0.f, 0.f, 0.f, 0.f);
    if (a.dh_extra) {
      const float4 x4 = *reinterpret_cast<const float4 *>(a.dh_extra + (size_t)m * a.dh_extra_ld + e);
      d4.x += x4.x; d4.y += x4.y; d4.z += x4.z; d4.w += x4.w;
    }
    const float dd[4] = {d4.x, d4.y, d4.z, d4.w}, rg[4] = {r4.x, r4.y, r4.z, r4.w}, ug[4] = {u4.x, u4.y, u4.z, u4.w};
    const float ng[4] = {n4.x, n4.y, n4.z, n4.w}, an[4] = {a4.x, a4.y, a4.z, a4.w}, hp[4] = {h4.x, h4.y, h4.z, h4.w};
    float dar[4], dau[4], dan[4], danr[4], dhn[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const float dn = dd[c] * (1.0f - ug[c]), du = dd[c] * (hp[c] - ng[c]);
      dan[c] = dn * (1.0f - ng[c] * ng[c]);
      dau[c] = du * ug[c] * (1.0f - ug[c]);
      dar[c] = dan[c] * an[c] * rg[c] * (1.0f - rg[c]);
      danr[c] = dan[c] * rg[c];
      dhn[c] = dd[c] * ug[c];
      s_r[c] += dar[c]; s_u[c] += dau[c]; s_n[c] += dan[c]; s_nr[c] += danr[c];
    }
    if (a.dah32) {
      *reinterpret_cast<float4 *>(a.dah32 + g3) = make_float4(dar[0], dar[1], dar[2], dar[3]);
      *reinterpret_cast<float4 *>(a.dah32 + g3 + E) = make_float4(dau[0], dau[1], dau[2], dau[3]);
      *reinterpret_cast<float4 *>(a.dah32 + g3 + 2 * E) = make_float4(danr[0], danr[1], danr[2], danr[3]);
      *reinterpret_cast<float4 *>(a.dan32 + idx) = make_float4(dan[0], dan[1], dan[2], dan[3]);
    }
    if (dah_hi) {
      put4(dah_hi, dah_lo, g3, dar); put4(dah_hi, dah_lo, g3 + E, dau); put4(dah_hi, dah_lo, g3 + 2 * E, danr);
      put4(dan_hi, dan_lo, idx, dan);
    }
    *reinterpret_cast<float4 *>(a.dh + idx) = make_float4(dhn[0], dhn[1], dhn[2], dhn[3]);
  }
  // reduce the four sums over the block's row lanes, then one atomic per (unit, sum) and block
  float *q = red + (size_t)rl * E + e;
  const size_t plane = (size_t)rpb * E;
#pragma unroll
  for (int c = 0; c < 4; ++c) { q[c] = s_r[c]; q[plane + c] = s_u[c]; q[2 * plane + c] = s_n[c]; q[3 * plane + c] = s_nr[c]; }
  __syncthreads();
  for (int i = threadIdx.x; i < 4 * E; i += 256) {
    const int which = i / E, u = i - which * E;
    float s = 0.f;
    for (int r = 0; r < rpb; ++r) s += red[(size_t)which * plane + (size_t)r * E + u];
    if (kPart) part[(size_t)blockIdx.x * 4 * E + i] += s;
    else if (which == 0) { atomicAdd(a.gb_ih + u, s); atomicAdd(a.gb_hh + u, s); }
    else if (which == 1) { atomicAdd(a.gb_ih + E + u, s); atomicAdd(a.gb_hh + E + u, s); }
    else if (which == 2) atomicAdd(a.gb_ih + 2 * E + u, s);
    else atomicAdd(a.gb_hh + 2 * E + u, s);
  }
}

// Grids of the two enc_gate_bwd2 kernels: blocks of the vectorised kernel (0 when the shape does not fit it), and row
// strip / blocks of the scalar kernel.
static int bwd2_v4_blocks(int M, int E) {
  const int tpr = E / 4;
  if (E % 4 != 0 || tpr < 1 || tpr > 256 || 256 % tpr != 0) return 0;
  const int rpb = 256 / tpr;
  const int blocks = (M + rpb - 1) / rpb;
  return blocks > 148 * 6 ? 148 * 6 : blocks;
}
static int bwd2_scalar_rpb(int M, int E, int *threads, int *cb) {
  *threads = E >= 256 ? 256 : (E >= 128 ? 128 : 64);
  *cb = (E + *threads - 1) / *threads;
  int rpb = 32;
  while ((long)((M + rpb - 1) / rpb) * *cb > 148 * 16 && rpb < 4096) rpb *= 2;
  return rpb;
}

int enc_gate_bwd2_part_rows(int M, int E) {
  int threads, cb;
  const int rpb = bwd2_scalar_rpb(M, E, &threads, &cb), scalar = (M + rpb - 1) / rpb, v4 = bwd2_v4_blocks(M, E);
  return scalar > v4 ? scalar : v4;
}

int enc_gate_bwd2(const EncStepBwd2 &a, cudaStream_t st, float *part) {
  auto al16 = [](const void *p) { return p == nullptr || ((uintptr_t)p & 15) == 0; };
  const int v4 = bwd2_v4_blocks(a.M, a.E);
  if (v4 > 0 && al16(a.dh) && al16(a.gates) && al16(a.ahn) && al16(a.hprev) &&
      al16(a.dah32) && al16(a.dan32) && al16(a.dh_extra) && (a.dh_extra == nullptr || a.dh_extra_ld % 4 == 0) &&
      (((uintptr_t)a.dah_hi | (uintptr_t)a.dah_lo | (uintptr_t)a.dan_hi | (uintptr_t)a.dan_lo) & 7) == 0) {
    const size_t smem = (size_t)4 * (256 / (a.E / 4)) * a.E * sizeof(float);
    if (part) enc_gate_bwd2_v4_kernel<true><<<v4, 256, smem, st>>>(a, part);
    else enc_gate_bwd2_v4_kernel<false><<<v4, 256, smem, st>>>(a, nullptr);
    LFI_LAUNCH_CHECK();
    return LFI_OK;
  }
  int threads, cb;
  const int rpb = bwd2_scalar_rpb(a.M, a.E, &threads, &cb);
  const dim3 grid((a.M + rpb - 1) / rpb, cb);
  if (part) enc_gate_bwd2_kernel<true><<<grid, threads, 0, st>>>(a, rpb, part);
  else enc_gate_bwd2_kernel<false><<<grid, threads, 0, st>>>(a, rpb, nullptr);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

// Adjoint of gather_windows: thread = one element dx[b][tau][c]; the (t', s) pairs whose window reads frame tau are visited
// in increasing t', so every element is one thread's fixed-order sum (no atomics although windows overlap when Tp > 1).
// ADD: the term add[tau - t0] of frames t0 <= tau < t0 + Tp comes last.
template <bool ADD>
__global__ void window_grad_kernel(float *dx, const float *src, int ld, int layout_steps, const float *mask, int B, int T, int dim,
                                   int hist, int off, int t0, int Tp, const float *add) {
  const size_t M = (size_t)Tp * B;
  const size_t n = (size_t)B * T * dim;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % dim);
    const size_t q = e / dim;
    const int tau = (int)(q % T), b = (int)(q / T);
    float acc = 0.f;
    for (int tp = 0; tp < Tp; ++tp) {
      const int s = tau - t0 - tp + hist - off;
      if (s < 0 || s >= hist) continue;
      const size_t m = (size_t)tp * B + b;
      float v = layout_steps ? src[((size_t)s * M + m) * ld + c] : src[m * ld + (size_t)s * dim + c];
      if (mask) v *= mask[m * hist + s];
      acc += v;
    }
    if (ADD && tau >= t0 && tau < t0 + Tp) acc += add[((size_t)(tau - t0) * B + b) * dim + c];
    dx[e] = acc;
  }
}
int window_grad(float *dx, const float *src, int ld, int layout_steps, const float *mask, int B, int T, int dim, int hist, int off, int t0,
                int Tp, cudaStream_t st, const float *add) {
  if (add)
    window_grad_kernel<true><<<blocks_for((size_t)B * T * dim), TB, 0, st>>>(dx, src, ld, layout_steps, mask, B, T, dim, hist, off, t0, Tp, add);
  else
    window_grad_kernel<false><<<blocks_for((size_t)B * T * dim), TB, 0, st>>>(dx, src, ld, layout_steps, mask, B, T, dim, hist, off, t0, Tp, nullptr);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

// ------------------------------------------------------------------------------------------------
__global__ void lu_build_kernel(float *Lm, float *Um, const float *l, const float *u, const float *log_s, const float *sign_s, int K, int C) {
  const size_t n = (size_t)K * C * C;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const int j = (int)(e % C), i = (int)((e / C) % C), k = (int)(e / ((size_t)C * C));
    Lm[e] = i > j ? l[e] : (i == j ? 1.0f : 0.0f);
    Um[e] = i < j ? u[e] : (i == j ? sign_s[k * C + i] * expf(log_s[k * C + i]) : 0.0f);
  }
}
int lu_build(float *Lm, float *Um, const float *l, const float *u, const float *log_s, const float *sign_s, int K, int C, cudaStream_t st) {
  lu_build_kernel<<<blocks_for((size_t)K * C * C), TB, 0, st>>>(Lm, Um, l, u, log_s, sign_s, K, C);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

// Triangular inverses in fp64 (the reference inverts L and U with torch.inverse(x.double()).float(),
// modules.py:175-176).  Thread j solves column j by substitution; scratch holds the fp64 columns.
__global__ void tri_inverse_kernel(float *Linv, float *Uinv, double *scratch, const float *Lm, const float *Um, int C) {
  const int k = blockIdx.x, which = blockIdx.y, j = threadIdx.x;
  if (j >= C) return;
  const float *A = (which == 0 ? Lm : Um) + (size_t)k * C * C;
  float *out = (which == 0 ? Linv : Uinv) + (size_t)k * C * C;
  double *x = scratch + ((size_t)(k * 2 + which)) * C * C;  // x[i*C + j]
  if (which == 0) {
    for (int i = 0; i < C; ++i) {
      double s = (i == j) ? 1.0 : 0.0;
      for (int m = 0; m < i; ++m) s -= (double)A[i * C + m] * x[m * C + j];
      x[i * C + j] = s / (double)A[i * C + i];
    }
  } else {
    for (int i = C - 1; i >= 0; --i) {
      double s = (i == j) ? 1.0 : 0.0;
      for (int m = i + 1; m < C; ++m) s -= (double)A[i * C + m] * x[m * C + j];
      x[i * C + j] = s / (double)A[i * C + i];
    }
  }
  for (int i = 0; i < C; ++i) out[i * C + j] = (float)x[i * C + j];
}
int tri_inverse_f64(float *Linv, float *Uinv, double *scratch, const float *Lm, const float *Um, int K, int C, cudaStream_t st) {
  tri_inverse_kernel<<<dim3(K, 2), round_up(C, 32), 0, st>>>(Linv, Uinv, scratch, Lm, Um, C);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

__global__ void lu_mask_grads_kernel(float *dl, float *du, float *dlog_s, const float *dL, const float *dU, const float *log_s,
                                     const float *sign_s, int K, int C) {
  const size_t n = (size_t)K * C * C;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const int j = (int)(e % C), i = (int)((e / C) % C), k = (int)(e / ((size_t)C * C));
    if (i > j) dl[e] += dL[e];
    if (i < j) du[e] += dU[e];
    if (i == j) dlog_s[k * C + i] += dU[e] * sign_s[k * C + i] * expf(log_s[k * C + i]);
  }
}
int lu_mask_grads(float *dl, float *du, float *dlog_s, const float *dL, const float *dU, const float *log_s, const float *sign_s,
                  int K, int C, cudaStream_t st) {
  lu_mask_grads_kernel<<<blocks_for((size_t)K * C * C), TB, 0, st>>>(dl, du, dlog_s, dL, dU, log_s, sign_s, K, C);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

// ------------------------------------------------------------------------------------------------
__global__ void sumsq_kernel(float *out, const float *g, size_t n) {
  __shared__ float part[TB / 32];
  float s = 0.f;
  const size_t n4 = n / 4;
  const float4 *g4 = reinterpret_cast<const float4 *>(g);
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n4; e += (size_t)gridDim.x * blockDim.x) {
    const float4 v = g4[e];
    s += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  for (size_t e = n4 * 4 + blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) s += g[e] * g[e];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < TB / 32 ? part[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) atomicAdd(out, v);
  }
}
int sumsq(float *out2, const float *g, size_t n, cudaStream_t st) {
  LFI_CUDA(cudaMemsetAsync(out2, 0, 2 * sizeof(float), st));
  sumsq_kernel<<<blocks_for(n / 4 + 1, TB, 148 * 4), TB, 0, st>>>(out2, g, n);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

namespace {
// the gradient's factor: grad_scale times the clip_grad_norm_ coefficient (max_norm / (norm + 1e-6), clamped to 1;
// max_norm <= 0: no clipping), norm = sqrt(sumsq) * grad_scale
__device__ __forceinline__ float clip_grad_scale(const float *sumsq_in, float grad_scale, float max_norm) {
  const float norm = sqrtf(sumsq_in[0]) * grad_scale;
  float coef = 1.0f;
  if (max_norm > 0.f) coef = fminf(max_norm / (norm + 1e-6f), 1.0f);
  return grad_scale * coef;
}
__device__ __forceinline__ float4 ld4_or0(const float *p, size_t e) {
  return p ? reinterpret_cast<const float4 *>(p)[e] : make_float4(0.f, 0.f, 0.f, 0.f);
}
__device__ __forceinline__ bool aligned16(const void *p) { return ((uintptr_t)p & 15) == 0; }
}  // namespace

// torch.nn.utils.clip_grad_norm_ (coef = max_norm / (norm + 1e-6), clamped to 1) followed by torch.optim.Adam
// (no weight decay, no amsgrad): the reference's configure_optimizers + gradient_clip_val.
__global__ void clip_adam_kernel(float *theta, const float *grad, float *m, float *v, size_t n, float lr, float b1, float b2,
                                 float omb1, float omb2, float eps, float max_norm, float grad_scale, float bc1,
                                 float bc2_sqrt, const float *sumsq_in, const float *hyper) {
  if (hyper) { lr = hyper[0]; bc1 = hyper[1]; bc2_sqrt = hyper[2]; }  // captured launches: the per-step scalars live on the device
  const float gs = clip_grad_scale(sumsq_in, grad_scale, max_norm);
  const float step = lr / bc1;
  auto upd = [&](float &th, float gr, float &mo, float &ve) {
    const float g = gr * gs;
    const float mm = b1 * mo + omb1 * g;
    const float vv = b2 * ve + omb2 * g * g;
    mo = mm; ve = vv;
    th -= step * mm / (sqrtf(vv) / bc2_sqrt + eps);
  };
  const bool vec = ((((uintptr_t)theta | (uintptr_t)grad | (uintptr_t)m | (uintptr_t)v) & 15) == 0);
  const size_t n4 = vec ? n / 4 : 0;  // 128-bit accesses over the aligned body (four streams in, three out: HBM bound)
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n4; e += (size_t)gridDim.x * blockDim.x) {
    float4 t4 = reinterpret_cast<float4 *>(theta)[e], m4 = reinterpret_cast<float4 *>(m)[e], v4 = reinterpret_cast<float4 *>(v)[e];
    const float4 g4 = reinterpret_cast<const float4 *>(grad)[e];
    upd(t4.x, g4.x, m4.x, v4.x); upd(t4.y, g4.y, m4.y, v4.y); upd(t4.z, g4.z, m4.z, v4.z); upd(t4.w, g4.w, m4.w, v4.w);
    reinterpret_cast<float4 *>(theta)[e] = t4; reinterpret_cast<float4 *>(m)[e] = m4; reinterpret_cast<float4 *>(v)[e] = v4;
  }
  for (size_t e = 4 * n4 + blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x)
    upd(theta[e], grad[e], m[e], v[e]);
}
int clip_adam(float *theta, const float *grad, float *m, float *v, size_t n, float lr, float b1, float b2, float eps,
              float max_norm, float grad_scale, int step, const float *sumsq_in, cudaStream_t st, const float *hyper) {
  // scalar coefficients in double, as torch.optim.Adam computes them on the host
  const double b1d = (double)b1, b2d = (double)b2;
  const float bc1 = (float)(1.0 - pow(b1d, (double)step));
  const float bc2s = (float)sqrt(1.0 - pow(b2d, (double)step));
  clip_adam_kernel<<<blocks_for((n + 3) / 4, TB, 148 * 8), TB, 0, st>>>(theta, grad, m, v, n, lr, b1, b2, (float)(1.0 - b1d),
                                                               (float)(1.0 - b2d), eps, max_norm, grad_scale, bc1, bc2s,
                                                               sumsq_in, hyper);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

// clip_grad_norm_ followed by torch.optim.SGD (single-tensor semantics).  hyper[0] = lr; hyper[1] != 0: the buffer holds no
// value yet (torch's first momentum step, buf = g), so it is written without being read.
__global__ void clip_sgd_kernel(float *theta, const float *grad, float *buf, size_t n, float momentum, float omd, float wd,
                                int nesterov, float max_norm, float grad_scale, const float *sumsq_in, const float *hyper) {
  const float lr = hyper[0];
  const bool first = hyper[1] != 0.f;
  const float gs = clip_grad_scale(sumsq_in, grad_scale, max_norm);
  auto upd = [&](float &th, float gr, float &bu) {
    float g = gr * gs;
    if (wd != 0.f) g += wd * th;
    if (buf) {
      bu = first ? g : momentum * bu + omd * g;
      g = nesterov ? g + momentum * bu : bu;
    }
    th -= lr * g;
  };
  const float *bin = first ? nullptr : buf;
  const bool vec = aligned16(theta) && aligned16(grad) && aligned16(buf);
  const size_t n4 = vec ? n / 4 : 0;  // 128-bit accesses over the aligned body
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n4; e += (size_t)gridDim.x * blockDim.x) {
    float4 t4 = reinterpret_cast<float4 *>(theta)[e], b4 = ld4_or0(bin, e);
    const float4 g4 = reinterpret_cast<const float4 *>(grad)[e];
    upd(t4.x, g4.x, b4.x); upd(t4.y, g4.y, b4.y); upd(t4.z, g4.z, b4.z); upd(t4.w, g4.w, b4.w);
    reinterpret_cast<float4 *>(theta)[e] = t4;
    if (buf) reinterpret_cast<float4 *>(buf)[e] = b4;
  }
  for (size_t e = 4 * n4 + blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    float bu = bin ? bin[e] : 0.f;
    upd(theta[e], grad[e], bu);
    if (buf) buf[e] = bu;
  }
}
int clip_sgd(float *theta, const float *grad, float *buf, size_t n, const float *hyper, float momentum, float dampening,
             float weight_decay, int nesterov, float max_norm, float grad_scale, const float *sumsq_in, cudaStream_t st) {
  clip_sgd_kernel<<<blocks_for((n + 3) / 4, TB, 148 * 8), TB, 0, st>>>(theta, grad, buf, n, momentum, (float)(1.0 - (double)dampening),
                                                                        weight_decay, nesterov, max_norm, grad_scale, sumsq_in, hyper);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

// clip_grad_norm_ followed by torch.optim.RMSprop (single-tensor semantics; grad_avg != nullptr: centered, buf != nullptr:
// momentum).  hyper[0] = lr.  The centered average moves as torch's lerp_ does (weight 1 - alpha).
__global__ void clip_rmsprop_kernel(float *theta, const float *grad, float *sq, float *ga, float *buf, size_t n, float alpha,
                                    float oma, float eps, float wd, float momentum, float max_norm, float grad_scale,
                                    const float *sumsq_in, const float *hyper) {
  const float lr = hyper[0];
  const float gs = clip_grad_scale(sumsq_in, grad_scale, max_norm);
  auto upd = [&](float &th, float gr, float &s, float &a, float &bu) {
    float g = gr * gs;
    if (wd != 0.f) g += wd * th;
    s = alpha * s + oma * g * g;
    float avg;
    if (ga) {
      a = oma < 0.5f ? a + oma * (g - a) : g - (g - a) * (1.0f - oma);
      avg = sqrtf(s - a * a) + eps;
    } else {
      avg = sqrtf(s) + eps;
    }
    if (buf) {
      bu = momentum * bu + g / avg;
      th -= lr * bu;
    } else {
      th -= lr * (g / avg);
    }
  };
  const bool vec = aligned16(theta) && aligned16(grad) && aligned16(sq) && aligned16(ga) && aligned16(buf);
  const size_t n4 = vec ? n / 4 : 0;  // 128-bit accesses over the aligned body
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n4; e += (size_t)gridDim.x * blockDim.x) {
    float4 t4 = reinterpret_cast<float4 *>(theta)[e], s4 = reinterpret_cast<float4 *>(sq)[e];
    float4 a4 = ld4_or0(ga, e), b4 = ld4_or0(buf, e);
    const float4 g4 = reinterpret_cast<const float4 *>(grad)[e];
    upd(t4.x, g4.x, s4.x, a4.x, b4.x); upd(t4.y, g4.y, s4.y, a4.y, b4.y);
    upd(t4.z, g4.z, s4.z, a4.z, b4.z); upd(t4.w, g4.w, s4.w, a4.w, b4.w);
    reinterpret_cast<float4 *>(theta)[e] = t4; reinterpret_cast<float4 *>(sq)[e] = s4;
    if (ga) reinterpret_cast<float4 *>(ga)[e] = a4;
    if (buf) reinterpret_cast<float4 *>(buf)[e] = b4;
  }
  for (size_t e = 4 * n4 + blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    float a = ga ? ga[e] : 0.f, bu = buf ? buf[e] : 0.f;
    upd(theta[e], grad[e], sq[e], a, bu);
    if (ga) ga[e] = a;
    if (buf) buf[e] = bu;
  }
}
int clip_rmsprop(float *theta, const float *grad, float *square_avg, float *grad_avg, float *buf, size_t n, const float *hyper,
                 float alpha, float eps, float weight_decay, float momentum, float max_norm, float grad_scale, const float *sumsq_in,
                 cudaStream_t st) {
  clip_rmsprop_kernel<<<blocks_for((n + 3) / 4, TB, 148 * 8), TB, 0, st>>>(theta, grad, square_avg, grad_avg, buf, n, alpha,
                                                                            (float)(1.0 - (double)alpha), eps, weight_decay, momentum,
                                                                            max_norm, grad_scale, sumsq_in, hyper);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

__global__ void fill_kernel(float *p, float v, size_t n) {
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) p[e] = v;
}
int fill(float *p, float v, size_t n, cudaStream_t st) {
  if (n == 0) return LFI_OK;
  fill_kernel<<<blocks_for(n), TB, 0, st>>>(p, v, n);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

// ------------------------------------------------------------------------------------------------
// column sums of split-bf16 planes (bias gradients of the flow-step RNN from the dG / dA_h operand planes):
// block = 16 column groups (4 bf16 each) x 16 row lanes, grid = (column blocks, row splits, batch); one atomic per column and block
__global__ void colsum_planes_kernel(float *out1, float *out2, int period, int lim2, long so, const __nv_bfloat16 *__restrict__ hi,
                                     const __nv_bfloat16 *__restrict__ lo, int ld, long sb, int rows, int col0, int cols, int rows_per_block) {
  __shared__ float part[16][65];
  const int cg = threadIdx.x & 15, rl = threadIdx.x >> 4;
  const int j0 = blockIdx.x * 64 + 4 * cg;
  const int b = blockIdx.z;
  const int r0 = blockIdx.y * rows_per_block, r1 = min(rows, r0 + rows_per_block);
  float s[4] = {0.f, 0.f, 0.f, 0.f};
  if (j0 < cols) {
    const __nv_bfloat16 *ph = hi + (size_t)b * sb + col0 + j0, *pl = lo ? lo + (size_t)b * sb + col0 + j0 : nullptr;
    for (int r = r0 + rl; r < r1; r += 16) {
      const uint2 h = *reinterpret_cast<const uint2 *>(ph + (size_t)r * ld);
      s[0] += __uint_as_float(h.x << 16); s[1] += __uint_as_float(h.x & 0xffff0000u);
      s[2] += __uint_as_float(h.y << 16); s[3] += __uint_as_float(h.y & 0xffff0000u);
      if (pl) {
        const uint2 l = *reinterpret_cast<const uint2 *>(pl + (size_t)r * ld);
        s[0] += __uint_as_float(l.x << 16); s[1] += __uint_as_float(l.x & 0xffff0000u);
        s[2] += __uint_as_float(l.y << 16); s[3] += __uint_as_float(l.y & 0xffff0000u);
      }
    }
  }
#pragma unroll
  for (int e = 0; e < 4; ++e) part[rl][4 * cg + e] = s[e];
  __syncthreads();
  if (threadIdx.x < 64) {
    const int j = blockIdx.x * 64 + threadIdx.x;
    if (j < cols) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) t += part[i][threadIdx.x];
      atomicAdd(out1 + (size_t)b * so + j, t);
      if (out2 && (j % period) < lim2) atomicAdd(out2 + (size_t)b * so + j, t);
    }
  }
}
int colsum_planes(float *out1, float *out2, int period, int lim2, long so, const void *hi, const void *lo, int ld, long sb, int batch, int rows,
                  int col0, int cols, cudaStream_t st) {
  if (rows <= 0 || cols <= 0 || batch <= 0) return LFI_OK;
  LFI_REQUIRE(cols % 4 == 0 && col0 % 4 == 0 && ld % 4 == 0 && sb % 4 == 0 && (((uintptr_t)hi | (uintptr_t)lo) & 7) == 0, LFI_ERR_ARG,
              "colsum_planes: planes must allow 8-byte accesses");
  const int cb = (cols + 63) / 64;
  int rb = (148 * 8 + cb * batch - 1) / (cb * batch);
  const int maxrb = (rows + 63) / 64;
  if (rb > maxrb) rb = maxrb;
  if (rb < 1) rb = 1;
  const int rpb = (rows + rb - 1) / rb;
  colsum_planes_kernel<<<dim3(cb, rb, batch), 256, 0, st>>>(out1, out2, period > 0 ? period : 1, lim2, so, (const __nv_bfloat16 *)hi,
                                                            (const __nv_bfloat16 *)lo, ld, sb, rows, col0, cols, rpb);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

// ------------------------------------------------------------------------------------------------
// generated frames -> 106-wide FLAME vectors (generate_motion_from_model.py:39-51, 68); thread = output element, coalesced
__global__ void expand_faces_kernel(const float *__restrict__ x, const float *__restrict__ means, const float *__restrict__ stds, size_t rows,
                                    int exp_dim, int jaw_dim, int neck_dim, float *__restrict__ out) {
  const int C = exp_dim + jaw_dim + neck_dim;
  const size_t total = rows * 106;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    const size_t r = e / 106;
    const int j = (int)(e - r * 106);
    int c = -1;
    if (j < exp_dim) c = j;
    else if (j >= 100 && j < 100 + jaw_dim) c = exp_dim + (j - 100);
    else if (j >= 103 && j < 103 + neck_dim) c = exp_dim + jaw_dim + (j - 103);
    float v = 0.f;
    if (c >= 0) {
      v = x[r * C + c];
      if (means) v = __fadd_rn(__fmul_rn(v, stds[c]), means[c]);  // torch: two rounded operations, no contraction
    }
    out[e] = v;
  }
}
int expand_faces(const float *x, const float *means, const float *stds, size_t rows, int exp_dim, int jaw_dim, int neck_dim, float *out,
                 cudaStream_t st) {
  if (rows == 0) return LFI_OK;
  expand_faces_kernel<<<blocks_for(rows * 106), TB, 0, st>>>(x, means, stds, rows, exp_dim, jaw_dim, neck_dim, out);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

// Validation metric of the reference (calc_jerk, glow/utils.py:53-58; mimicry_logger.py:175-184): mean |third difference| along
// time of [B, T, C].  The three differences are taken as three rounded fp32 subtractions, exactly as torch does; the sum runs
// in fp64 (per-block partial sums, one atomic per block), so the mean agrees with the reference's to fp32 rounding.
__global__ void jerk_kernel(const float *__restrict__ x, int B, int T, int C, double *__restrict__ acc) {
  const size_t n = (size_t)B * (T - 3) * C;
  double s = 0.0;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % C);
    const size_t q = e / C;
    const int t = (int)(q % (T - 3)), b = (int)(q / (T - 3));
    const float *p = x + ((size_t)b * T + t) * C + c;
    const float x0 = p[0], x1 = p[C], x2 = p[2 * (size_t)C], x3 = p[3 * (size_t)C];
    const float d0 = __fsub_rn(x1, x0), d1 = __fsub_rn(x2, x1), d2 = __fsub_rn(x3, x2);
    const float a0 = __fsub_rn(d1, d0), a1 = __fsub_rn(d2, d1);
    s += (double)fabsf(__fsub_rn(a1, a0));
  }
  __shared__ double red[TB / 32];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < TB / 32; ++i) t += red[i];
    atomicAdd(acc, t);
  }
}
__global__ void jerk_finish_kernel(const double *acc, double n, float *out) { out[0] = (float)(acc[0] / n); }
int jerk(const float *x, int B, int T, int C, double *scratch, float *out, cudaStream_t st) {
  LFI_CUDA(cudaMemsetAsync(scratch, 0, sizeof(double), st));
  const size_t n = (size_t)B * (T - 3) * C;
  jerk_kernel<<<blocks_for(n), TB, 0, st>>>(x, B, T, C, scratch);
  jerk_finish_kernel<<<1, 1, 0, st>>>(scratch, (double)n, out);
  LFI_LAUNCH_CHECK_N(2);
  return LFI_OK;
}

// Input side (SURVEY.md section 8(f) rank 4): MimicryDataset.__getitem__ + the DataLoader's collate (mimicry_data_module.py:44-78)
// on a corpus that is resident in HBM.  raw [rows, dim] holds every segment of one modality back to back; window b of the
// batch is the T consecutive rows starting at row0[b]: out[b][t][:] = raw[row0[b] + t][:].  Pure copy (bit exact), 128-bit
// accesses when dim % 4 == 0 and the bases are 16-byte aligned.
__global__ void gather_batch_kernel(const float *__restrict__ raw, const long long *__restrict__ row0, int B, int T, int dim, float *__restrict__ out) {
  const size_t n = (size_t)B * T * dim;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const size_t per = (size_t)T * dim;
    const int b = (int)(e / per);
    out[e] = raw[(size_t)row0[b] * dim + (e - (size_t)b * per)];
  }
}
__global__ void gather_batch_v4_kernel(const float4 *__restrict__ raw, const long long *__restrict__ row0, int B, int T, int dim4, float4 *__restrict__ out) {
  const size_t n = (size_t)B * T * dim4;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const size_t per = (size_t)T * dim4;
    const int b = (int)(e / per);
    out[e] = raw[(size_t)row0[b] * dim4 + (e - (size_t)b * per)];
  }
}
int gather_batch(const float *raw, const long long *row0, int B, int T, int dim, float *out, cudaStream_t st) {
  if (dim % 4 == 0 && (((uintptr_t)raw | (uintptr_t)out) & 15) == 0) {
    gather_batch_v4_kernel<<<blocks_for((size_t)B * T * (dim / 4)), TB, 0, st>>>((const float4 *)raw, row0, B, T, dim / 4, (float4 *)out);
  } else {
    gather_batch_kernel<<<blocks_for((size_t)B * T * dim), TB, 0, st>>>(raw, row0, B, T, dim, out);
  }
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

}  // namespace aux
}  // namespace lfi
