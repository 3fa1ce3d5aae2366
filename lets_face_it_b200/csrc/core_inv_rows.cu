// Inverse flow core for sampling with the gate-ih pre-activations given (FlowStep.reverse_flow, models.py:345-373,
// driven by SeqGlow.inference / SeqGlow.invert, models.py:567-645).
//
// A sampling launch holds few sequences per SM (1024 sequences / 148 SMs), so the tile-GEMM scheme of the wavefront
// kernels (weights staged through shared memory for a tile of rows) spends its time on staging and barriers.  Here a
// CTA owns RR sequences and ONE THREAD OWNS ONE GATE COLUMN of [W_ih[:, :Ci] ; W_hh]: the RR activation values of each
// reduction index are broadcast from shared memory and every weight element is read by exactly one thread.  The
// per-step weights (272 KB at final_model.yaml, L2 resident) are streamed by the bulk-copy engine (cp.async.bulk +
// mbarrier transaction counts) through a ring of three 48 KB slots, always three chunks ahead of the math, across
// step and frame boundaries; the small products (LinearZeros, 1x1 conv inverse) split their reduction over thread groups.
#include "core_api.cuh"

namespace lfi {
namespace core {

template <int RR> struct RowVec;
template <> struct RowVec<8> {
  static __device__ __forceinline__ void load(float (&a)[8], const float *p) {
    const float4 u = *reinterpret_cast<const float4 *>(p), v = *reinterpret_cast<const float4 *>(p + 4);
    a[0] = u.x; a[1] = u.y; a[2] = u.z; a[3] = u.w; a[4] = v.x; a[5] = v.y; a[6] = v.z; a[7] = v.w;
  }
};
template <> struct RowVec<4> {
  static __device__ __forceinline__ void load(float (&a)[4], const float *p) {
    const float4 u = *reinterpret_cast<const float4 *>(p);
    a[0] = u.x; a[1] = u.y; a[2] = u.z; a[3] = u.w;
  }
};

constexpr int RB_ROWS = 32;   // reduction rows of W_hh per streamed chunk
constexpr int RB_N = 3;       // chunks in flight
struct RowsPlan { int ring, chunk, Si, Sh, hs, zs, xs, part, vec, ld, bars, total; };
__host__ __device__ inline RowsPlan plan_rows(const Dims &d, int RR) {
  RowsPlan p;
  int o = 0;
  auto take = [&](int n) { int r = o; o += round_up(n, 4); return r; };
  const int Cm = d.Co > d.C ? d.Co : d.C;
  p.chunk = RB_ROWS * d.GH;     // floats per ring slot
  p.ring = take(RB_N * p.chunk);  // per-step weights streamed by the bulk-copy engine (cp.async.bulk + mbarrier)
  p.Si = take(RR * d.GH);       // [RR][GH] i-side gate pre-activations (z1 part + given G)
  p.Sh = take(RR * d.GH);       // [RR][GH] h-side gate pre-activations (+ b_hh)
  p.hs = take(d.H * RR);        // [H][RR]  state
  p.zs = take(d.C * RR);        // [C][RR]  current z (input of the inverse step)
  p.xs = take(d.C * RR);        // [C][RR]  after the inverse coupling
  p.part = take(4 * RR * Cm);   // [4][RR][Cm] partial sums of the split reductions
  p.vec = take(2 * d.C + 2 * d.Co);  // exp(-logs), bias, bf, exp(3 lf) of the current step
  p.ld = take(RR);
  p.bars = take(2 * RB_N);      // RB_N 64-bit mbarriers
  p.total = o;
  return p;
}

__device__ __forceinline__ unsigned smem_addr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init_(unsigned long long *bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait_(unsigned long long *bar, unsigned parity) {
  unsigned ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_addr(bar)), "r"(parity)
        : "memory");
  }
}
// one elected thread: announce the byte count, then hand the copy to the bulk-copy engine
__device__ __forceinline__ void bulk_load(float *dst, const float *src, unsigned bytes, unsigned long long *bar) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_addr(dst)), "l"(src), "r"(bytes), "r"(smem_addr(bar))
               : "memory");
}

// STASH: also store the activations of the step (InvArgs.st_x1 ...; one frame, one step); the instantiation without it is the
// plain inverse
template <int RR, bool STASH>
__global__ void core_inv_rows(InvArgs a) {
  extern __shared__ __align__(16) float sm[];
  const Dims &d = a.d;
  const int tid = threadIdx.x, NTH = blockDim.x;
  const int row0 = blockIdx.x * RR, nrows = min(RR, a.B - row0);
  const int C = d.C, Ci = d.Ci, Cz = d.Cz, Co = d.Co, H = d.H, GH = d.GH, B = a.B;
  const int Cm = Co > C ? Co : C;
  const RowsPlan pl = plan_rows(d, RR);
  float *Si = sm + pl.Si, *Sh = sm + pl.Sh, *hs = sm + pl.hs, *zs = sm + pl.zs, *xs = sm + pl.xs, *part = sm + pl.part;
  float *einv = sm + pl.vec, *anb = einv + C, *bfs = anb + C, *e3 = bfs + Co, *ldacc = sm + pl.ld;
  const int j = tid;  // gate column owned by this thread (j < GH)
  float *ring = sm + pl.ring;
  unsigned long long *bars = reinterpret_cast<unsigned long long *>(sm + pl.bars);
  // weight stream: per step the chunks [W_ih[:, :Ci]^T | W_hh^T in blocks of 32 reduction rows | Wf^T | W^-1], in the
  // order they are consumed, through a ring of RB_N slots; chunk g lives in slot g % RB_N
  const int nhh = H / RB_ROWS, nchunk = nhh + 3, nk = a.k_hi - a.k_lo + 1;
  const int total_chunks = a.Tc * nk * nchunk;
  auto issue = [&](int g) {  // thread 0 only
    const int si = g / nchunk, c = g - si * nchunk;
    const int k = a.k_hi - si % nk;
    const StepWeights w = a.dv.step(d, k);
    const float *src; unsigned bytes;
    if (c == 0) { src = w.WzT; bytes = (unsigned)(Ci * GH * 4); }
    else if (c <= nhh) { src = w.WhhT + (size_t)(c - 1) * RB_ROWS * GH; bytes = (unsigned)(RB_ROWS * GH * 4); }
    else if (c == nhh + 1) { src = w.WfT; bytes = (unsigned)(H * d.Cop * 4); }
    else { src = w.Winv; bytes = (unsigned)(C * d.Cp * 4); }
    bulk_load(ring + (g % RB_N) * pl.chunk, src, bytes, &bars[g % RB_N]);
  };
  if (tid == 0) {
    for (int b = 0; b < RB_N; ++b) mbar_init_(&bars[b], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (tid == 0)
    for (int g = 0; g < RB_N && g < total_chunks; ++g) issue(g);
  int gc = 0;  // next chunk to consume
  auto acquire = [&]() -> const float * {
    mbar_wait_(&bars[gc % RB_N], (unsigned)((gc / RB_N) & 1));
    return ring + (gc % RB_N) * pl.chunk;
  };
  auto release = [&]() {  // call after a __syncthreads that follows the last read of the slot
    if (tid == 0 && gc + RB_N < total_chunks) issue(gc + RB_N);
    ++gc;
  };

  for (int tc = 0; tc < a.Tc; ++tc) {
    // latent of this frame (GaussianDiag.sample output, models.py:511) or the given z (invert)
    for (int e = tid; e < RR * C; e += NTH) {
      const int r = e / C, c = e - r * C;
      zs[c * RR + r] = (r < nrows && a.noise) ? a.noise[((size_t)(a.t_rel0 + tc) * B + row0 + r) * C + c] : 0.f;
    }
    if (tid < RR) ldacc[tid] = 0.f;
    for (int k = a.k_hi; k >= a.k_lo; --k) {
      const StepWeights w = a.dv.step(d, k);
      // ---- prefetch: given gate-ih pre-activations, state, per-step vectors ------------------------------------------
      float gv[RR];
      if (j < GH) {
        const float *Gp = a.G + ((size_t)tc * B + row0) * a.g_ld + (size_t)(k - a.g_k0) * GH + j;
#pragma unroll
        for (int r = 0; r < RR; ++r) gv[r] = r < nrows ? __ldg(Gp + (size_t)r * a.g_ld) : 0.f;
      }
      for (int e = tid; e < RR * H; e += NTH) {
        const int r = e / H, m = e - r * H;
        hs[m * RR + r] = r < nrows ? a.hstate[((size_t)k * B + row0 + r) * H + m] : 0.f;
      }
      for (int e = tid; e < C; e += NTH) { einv[e] = expf(-w.an_logs[e]); anb[e] = w.an_bias[e]; }
      for (int e = tid; e < Co; e += NTH) { bfs[e] = w.bf[e]; e3[e] = expf(3.0f * w.lf[e]); }
      __syncthreads();
      // ---- 1. gate pre-activations: column j of [z1 ; h] . [W_ih[:, :Ci] ; W_hh]^T ------------------------------------
      float ai[RR], ah[RR];
#pragma unroll
      for (int r = 0; r < RR; ++r) { ai[r] = gv[r]; ah[r] = 0.f; }
      {
        const float *wz = acquire();
        if (j < GH) {
#pragma unroll 4
          for (int kk = 0; kk < Ci; ++kk) {
            const float wv = wz[kk * GH + j];
            float av[RR];
            RowVec<RR>::load(av, zs + kk * RR);
#pragma unroll
            for (int r = 0; r < RR; ++r) ai[r] = fmaf(av[r], wv, ai[r]);
          }
        }
        __syncthreads();
        release();
      }
      for (int cb = 0; cb < nhh; ++cb) {
        const float *wh = acquire();
        if (j < GH) {
#pragma unroll 8
          for (int kk = 0; kk < RB_ROWS; ++kk) {
            const float wv = wh[kk * GH + j];
            float av[RR];
            RowVec<RR>::load(av, hs + (cb * RB_ROWS + kk) * RR);
#pragma unroll
            for (int r = 0; r < RR; ++r) ah[r] = fmaf(av[r], wv, ah[r]);
          }
          if (cb == nhh - 1) {
            const float bh = w.b_hh[j];
#pragma unroll
            for (int r = 0; r < RR; ++r) { Si[r * GH + j] = ai[r]; Sh[r * GH + j] = ah[r] + bh; }
          }
        }
        __syncthreads();
        release();
      }
      // ---- 2. GRU gate math (nn.GRUCell, gate order r, z, n); new state to shared memory and to the carried state -------
      for (int e = tid; e < RR * H; e += NTH) {
        const int r = e / H, m = e - r * H;
        const float *si = Si + r * GH, *sh = Sh + r * GH;
        const float rg = fast_sigmoid(si[m] + sh[m]), ug = fast_sigmoid(si[H + m] + sh[H + m]);
        const float ng = fast_tanh(si[2 * H + m] + rg * sh[2 * H + m]);
        const float hp = hs[m * RR + r];
        const float hn = ng + ug * (hp - ng);
        hs[m * RR + r] = hn;
        if (r < nrows) a.hstate[((size_t)k * B + row0 + r) * H + m] = hn;
        if (STASH && r < nrows) {
          float *g = a.st_gates + (size_t)(row0 + r) * GH;
          g[m] = rg; g[H + m] = ug; g[2 * H + m] = ng;
          a.st_ahn[(size_t)(row0 + r) * H + m] = sh[2 * H + m];
        }
      }
      __syncthreads();
      // ---- 3. LinearZeros (modules.py:93-95): reduction split over 4 thread groups --------------------------------------
      {
        const float *wfs = acquire();
        const int jj = tid % Cm, kg = tid / Cm;
        if (kg < 4 && jj < Co) {
          float o[RR];
#pragma unroll
          for (int r = 0; r < RR; ++r) o[r] = 0.f;
          const int k0 = kg * (H / 4), k1 = kg == 3 ? H : k0 + H / 4;
          const float *wf = wfs + jj;
#pragma unroll 8
          for (int kk = k0; kk < k1; ++kk) {
            const float wv = wf[kk * d.Cop];
            float av[RR];
            RowVec<RR>::load(av, hs + kk * RR);
#pragma unroll
            for (int r = 0; r < RR; ++r) o[r] = fmaf(av[r], wv, o[r]);
          }
#pragma unroll
          for (int r = 0; r < RR; ++r) part[(kg * RR + r) * Cm + jj] = o[r];
        }
      }
      __syncthreads();
      release();
      // ---- 4. inverse coupling (models.py:358-366): z2 = z2 / scale - shift ---------------------------------------------
      for (int e = tid; e < RR * Cz; e += NTH) {
        const int r = e / Cz, q = e - r * Cz;
        auto osum = [&](int jj) {
          return (part[(0 * RR + r) * Cm + jj] + part[(1 * RR + r) * Cm + jj] + part[(2 * RR + r) * Cm + jj] + part[(3 * RR + r) * Cm + jj] + bfs[jj]) * e3[jj];
        };
        const float z2 = zs[(Ci + q) * RR + r];
        float v;
        if (d.affine) {
          const float shift = osum(2 * q), sc = osum(2 * q + 1);
          const float s = fmaxf(sigmoidf_(sc + 2.0f), d.eps);
          v = z2 / s - shift;
          if (a.logdet_out) atomicAdd(&ldacc[r], -logf(s));
        } else {
          v = z2 - osum(q);
        }
        xs[(Ci + q) * RR + r] = v;
        if (STASH && r < nrows) a.st_zc[(size_t)(row0 + r) * C + Ci + q] = v;
      }
      for (int e = tid; e < RR * Ci; e += NTH) {
        const int r = e / Ci, c = e - r * Ci;
        xs[c * RR + r] = zs[c * RR + r];
        if (STASH && r < nrows) a.st_zc[(size_t)(row0 + r) * C + c] = zs[c * RR + r];
      }
      // o as a loop of its own: a stored product inside the loop above would no longer contract into its FMAs, and the
      // coupling output would differ in the last bit from the plain instantiation's
      if (STASH)
        for (int e = tid; e < nrows * Co; e += NTH) {
          const int r = e / Co, jj = e - r * Co;
          a.st_o[(size_t)(row0 + r) * Co + jj] = (part[(0 * RR + r) * Cm + jj] + part[(1 * RR + r) * Cm + jj] + part[(2 * RR + r) * Cm + jj] +
                                                  part[(3 * RR + r) * Cm + jj] + bfs[jj]) * e3[jj];
        }
      __syncthreads();
      // ---- 5. 1x1 conv inverse, ActNorm inverse (modules.py:175-177, 189-193, 76-78) ----------------------------------------
      {
        const float *wis = acquire();
        const int jj = tid % Cm, kg = tid / Cm;
        if (kg < 4 && jj < C) {
          float o[RR];
#pragma unroll
          for (int r = 0; r < RR; ++r) o[r] = 0.f;
          const int per = (C + 3) / 4, k0 = kg * per, k1 = min(C, k0 + per);
          const float *wi = wis + jj;
#pragma unroll 4
          for (int kk = k0; kk < k1; ++kk) {
            const float wv = wi[kk * d.Cp];
            float av[RR];
            RowVec<RR>::load(av, xs + kk * RR);
#pragma unroll
            for (int r = 0; r < RR; ++r) o[r] = fmaf(av[r], wv, o[r]);
          }
#pragma unroll
          for (int r = 0; r < RR; ++r) part[(kg * RR + r) * Cm + jj] = o[r];
        }
      }
      __syncthreads();
      release();
      for (int e = tid; e < RR * C; e += NTH) {
        const int r = e / C, c = e - r * C;
        const float v = part[(0 * RR + r) * Cm + c] + part[(1 * RR + r) * Cm + c] + part[(2 * RR + r) * Cm + c] + part[(3 * RR + r) * Cm + c];
        if (STASH && r < nrows) a.st_x1[(size_t)(row0 + r) * C + c] = v;
        zs[c * RR + r] = v * einv[c] - anb[c];
      }
      __syncthreads();
    }
    // emit the frame
    const int t_abs = a.t_abs0 + tc;
    for (int e = tid; e < nrows * C; e += NTH) {
      const int r = e / C, c = e - r * C;
      a.faces_out[(size_t)(row0 + r) * a.fo_sb + (size_t)t_abs * a.fo_st + c] = zs[c * RR + r];
    }
    if (a.logdet_out && tid < nrows) a.logdet_out[(size_t)(a.t_rel0 + tc) * B + row0 + tid] = ldacc[tid];
    __syncthreads();
  }
}

bool inv_rows_supported(const InvArgs &a) {
  const Dims &d = a.d;
  if (a.cstatic || !a.G || d.G != 3) return false;
  const int Cm = d.Co > d.C ? d.Co : d.C;
  const int nth = round_up(d.GH, 32);
  if (d.H % RB_ROWS != 0 || d.Ci > RB_ROWS || d.H * d.Cop > RB_ROWS * d.GH || d.C * d.Cp > RB_ROWS * d.GH) return false;
  if (plan_rows(d, 4).total * (int)sizeof(float) > 227 * 1024) return false;
  return nth <= 1024 && 4 * Cm <= nth && d.H % 4 == 0;
}

template <int RR> static int launch_inv_rows_t(const InvArgs &a, cudaStream_t st) {
  const int bytes = plan_rows(a.d, RR).total * (int)sizeof(float);
  auto kern = a.st_x1 ? core_inv_rows<RR, true> : core_inv_rows<RR, false>;
  if (bytes > 48 * 1024) LFI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  kern<<<(a.B + RR - 1) / RR, round_up(a.d.GH, 32), bytes, st>>>(a);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

int launch_inv_rows(const InvArgs &a, cudaStream_t st) {
  const int rr = ((a.B + 7) / 8 >= 120 && plan_rows(a.d, 8).total * (int)sizeof(float) <= 227 * 1024) ? 8 : 4;
  return rr == 8 ? launch_inv_rows_t<8>(a, st) : launch_inv_rows_t<4>(a, st);
}

}  // namespace core
}  // namespace lfi
