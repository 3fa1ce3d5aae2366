// Sequential flow core, backward direction: reverse wavefronts over the (step k, frame t) cells.
// Cell (k,t) consumes d(output of step k) from cell (k+1,t) and d(h[k][t]) from cell (k,t+1) (BPTT of the
// coupling RNN, models.py:193-214) and produces d(input of step k), d(h[k][t-1]), the gate gradients dA_i /
// dA_h (whose weight gradients are taken afterwards as time-parallel GEMMs over the stash) and the small
// per-channel gradients (ActNorm bias/logs, b_hh, LinearZeros bias/logs) by per-CTA column sums + atomics.
#include "core_api.cuh"
#include "core_pipe.cuh"

namespace lfi {
namespace core {

// DXIN: the cells (0, t) also store the gradient of the flow input (BwdArgs.dx_in); the instantiation without it is the plain backward
template <int RPT, int KC, bool DXIN>
__global__ void __launch_bounds__(NT) core_bwd_wave(BwdArgs a, int wave, int kmin) {
  extern __shared__ __align__(16) float sm[];
  constexpr int R = Tile<RPT>::R, RS = Tile<RPT>::RS;
  const Dims &d = a.d;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int k = kmin + blockIdx.y, t = wave - k;
  const int row0 = blockIdx.x * R, nrows = min(R, a.B - row0);
  const int C = d.C, Ci = d.Ci, Cz = d.Cz, Co = d.Co, H = d.H, GH = d.GH, B = a.B, Tp = a.Tp;
  const bool gru = d.G == 3;
  const SmemPlan sp = plan_smem(d, R, true, false, KC);
  const StepWeights w = a.dv.step(d, k);
  const size_t cell = (size_t)k * Tp + t;
  const int pC = odd(C), pO = odd(Co > C ? Co : C), pS = odd(GH), pH = odd(H);
  float *xs = sm + sp.xs, *zact = sm + sp.zact, *zrow = sm + sp.zrow, *hp = sm + sp.hp, *cp = sm + sp.cp;
  float *S = sm + sp.S, *ahn = sm + sp.ahn, *orow = sm + sp.orow, *dact = sm + sp.dact, *dxr = sm + sp.dxr;
  float *dhr = sm + sp.dhr, *prod = sm + sp.prod, *cn = sm + sp.cn, *dldr = sm + sp.ldacc;

  // ---- A. loads ---------------------------------------------------------------------------------
  for (int e = tid; e < R * C; e += NT) {
    const int r = e / C, c = e - r * C;
    float dxo = 0.f, zf = 0.f;
    if (r < nrows) {
      const int b = row0 + r;
      zf = a.st.zf[(cell * B + b) * C + c];
      if (a.single >= 0) dxo = a.dz_ext[(size_t)b * C + c];
      else if (k == d.K - 1) dxo = a.dnll[(size_t)t * B + b] * a.z[((size_t)t * B + b) * C + c] / kLn2;  // d nll / d z = z / ln2
      else dxo = a.dx[((cell + Tp) * B + b) * C + c];
    }
    dxr[r * pC + c] = dxo;
    zrow[r * pC + c] = zf;
  }
  for (int e = tid; e < R * Co; e += NT) {
    const int r = e / Co, j = e - r * Co;
    orow[r * pO + j] = (r < nrows) ? a.st.o[(cell * B + row0 + r) * Co + j] : 0.f;
  }
  if (tid < R) {
    float v = 0.f;
    if (tid < nrows) {
      if (a.single >= 0) v = a.dld_ext ? a.dld_ext[row0 + tid] : 0.f;
      else v = -a.dnll[(size_t)t * B + row0 + tid] / kLn2;  // d nll / d logdet
    }
    dldr[tid] = v;
  }
  for (int r0 = 0; r0 < R; r0 += 4)  // four rows in flight per thread
    for (int j = tid; j < GH; j += NT) {
      float g[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) g[i] = (r0 + i < nrows) ? __ldg(a.st.gates + (cell * B + row0 + r0 + i) * GH + j) : 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) S[(r0 + i) * pS + j] = g[i];
    }
  for (int r0 = 0; r0 < R; r0 += 4)  // four rows requested per thread before the first is used
    for (int m = tid; m < H; m += NT) {
      float hv[4], cv[4], cnv[4], an[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = r0 + i;
        hv[i] = 0.f; cv[i] = 0.f; cnv[i] = 0.f; an[i] = 0.f;
        if (r < nrows) {
          const size_t idx = (cell * B + row0 + r) * H + m;
          if (t > 0) {
            hv[i] = a.st.h[idx - (size_t)B * H];
            if (!gru) cv[i] = a.st.c[idx - (size_t)B * H];
          } else if (a.single >= 0) {  // module API: the state the cell started from is given
            const size_t e1 = (size_t)(row0 + r) * H + m;
            if (a.h_prev_ext) hv[i] = a.h_prev_ext[e1];
            if (!gru && a.c_prev_ext) cv[i] = a.c_prev_ext[e1];
          }
          if (gru) {
            an[i] = a.st.ahn[idx];
          } else {
            cnv[i] = a.st.c[idx];
            if (a.single >= 0) an[i] = a.dc_ext ? a.dc_ext[(size_t)(row0 + r) * H + m] : 0.f;
            else an[i] = (t < Tp - 1) ? a.dc[idx + (size_t)B * H] : 0.f;  // dc flowing back from cell (k, t+1)
          }
        }
      }
      *reinterpret_cast<float4 *>(hp + m * RS + r0) = make_float4(hv[0], hv[1], hv[2], hv[3]);
#pragma unroll
      for (int i = 0; i < 4; ++i) ahn[(r0 + i) * pH + m] = an[i];
      if (!gru) {
        *reinterpret_cast<float4 *>(cp + m * RS + r0) = make_float4(cv[0], cv[1], cv[2], cv[3]);
        *reinterpret_cast<float4 *>(cn + m * RS + r0) = make_float4(cnv[0], cnv[1], cnv[2], cnv[3]);
      }
    }
  __syncthreads();

  // ---- B. coupling backward (models.py:331-341) ---------------------------------------------------
  for (int r = warp; r < R; r += NT / 32) {
    const float dld = dldr[r];
    for (int q = lane; q < Cz; q += 32) {
      const float dz2n = dxr[r * pC + Ci + q];
      if (d.affine) {
        const float shift = orow[r * pO + 2 * q], sc = orow[r * pO + 2 * q + 1];
        const float sg = sigmoidf_(sc + 2.0f), s = fmaxf(sg, d.eps);
        const float z2 = zrow[r * pC + Ci + q];
        const float ds = dz2n * (z2 + shift) + dld / s;
        const float dz2 = dz2n * s;
        const float dsc = (sg >= d.eps) ? ds * sg * (1.0f - sg) : 0.f;
        prod[r * pO + 2 * q] = dz2 * shift;
        prod[r * pO + 2 * q + 1] = dsc * sc;
        orow[r * pO + 2 * q] = dz2;
        orow[r * pO + 2 * q + 1] = dsc;
        xs[(2 * q) * RS + r] = dz2 * expf(3.0f * w.lf[2 * q]);
        xs[(2 * q + 1) * RS + r] = dsc * expf(3.0f * w.lf[2 * q + 1]);
        zrow[r * pC + Ci + q] = dz2;
      } else {
        prod[r * pO + q] = dz2n * orow[r * pO + q];
        orow[r * pO + q] = dz2n;
        xs[q * RS + r] = dz2n * expf(3.0f * w.lf[q]);
        zrow[r * pC + Ci + q] = dz2n;
      }
    }
    for (int c = lane; c < Ci; c += 32) zrow[r * pC + c] = dxr[r * pC + c];
  }
  __syncthreads();
  // dlin stash (= dO * e3, for dWf) + LinearZeros bias/logs gradients
  // (o = (lin + bf) * e3  =>  d bf = e3 * sum dO, d lf = 3 * sum dO*o)
  for (int e = tid; e < nrows * Co; e += NT) {
    const int r = e / Co, j = e - r * Co;
    a.dO[(cell * B + row0 + r) * Co + j] = xs[j * RS + r];
  }
  for (int j = tid; j < Co; j += NT) {
    float s1 = 0.f, s2 = 0.f;
    for (int r = 0; r < nrows; ++r) { s1 += orow[r * pO + j]; s2 += prod[r * pO + j]; }
    atomicAdd(&a.g_bf[(size_t)k * Co + j], s1 * expf(3.0f * w.lf[j]));
    atomicAdd(&a.g_lf[(size_t)k * Co + j], 3.0f * s2);
  }

  // ---- E. dh = dlin @ Wf (+ dh from the next frame) ------------------------------------------------
  tile_gemm<RPT, KC>(xs, w.Wf, H, Co, H, sm + sp.wst, [&](int r, int j, float v) {
    if (r < nrows) {
      if (a.single >= 0) { if (a.dh_ext) v += a.dh_ext[(size_t)(row0 + r) * H + j]; }
      else if (t < Tp - 1) v += a.dh[((cell + 1) * B + row0 + r) * H + j];
    }
    dhr[r * pH + j] = v;
  });
  __syncthreads();

  // ---- G. gate backward ------------------------------------------------------------------------------
  for (int e = tid; e < R * H; e += NT) {
    const int r = e % R, m = e / R;
    float *s = S + r * pS;
    const float dh = dhr[r * pH + m];
    if (gru) {
      const float rg = s[m], ug = s[H + m], ng = s[2 * H + m], hpv = hp[m * RS + r], an = ahn[r * pH + m];
      const float dn = dh * (1.0f - ug), du = dh * (hpv - ng);
      const float dan = dn * (1.0f - ng * ng), dau = du * ug * (1.0f - ug), dar = dan * an * rg * (1.0f - rg);
      s[m] = dar; s[H + m] = dau; s[2 * H + m] = dan;
      ahn[r * pH + m] = dan * rg;
      dact[m * RS + r] = dar; dact[(H + m) * RS + r] = dau; dact[(2 * H + m) * RS + r] = dan;
      dact[(GH + m) * RS + r] = dan * rg;
      dhr[r * pH + m] = dh * ug;
    } else {
      const float ig = s[m], fg = s[H + m], gg = s[2 * H + m], og = s[3 * H + m];
      const float tc = tanhf(cn[m * RS + r]);
      const float dc = dh * og * (1.0f - tc * tc) + ahn[r * pH + m];
      const float dai = dc * gg * ig * (1.0f - ig), daf = dc * cp[m * RS + r] * fg * (1.0f - fg);
      const float dag = dc * ig * (1.0f - gg * gg), dao = dh * tc * og * (1.0f - og);
      s[m] = dai; s[H + m] = daf; s[2 * H + m] = dag; s[3 * H + m] = dao;
      dact[m * RS + r] = dai; dact[(H + m) * RS + r] = daf; dact[(2 * H + m) * RS + r] = dag;
      dact[(3 * H + m) * RS + r] = dao;
      ahn[r * pH + m] = dc * fg;
      dhr[r * pH + m] = 0.f;
    }
  }
  __syncthreads();
  // dA_i -> dG (time-parallel backward + db_ih), dA_h stash (dW_hh), db_hh, LSTM dc_prev
  {
    const size_t gld = a.dg_ld ? (size_t)a.dg_ld : (size_t)d.K * GH;
    for (int r = 0; r < nrows; ++r)
      for (int j = tid; j < GH; j += NT) {
        const float vi = S[r * pS + j];
        const float vh = (gru && j >= 2 * H) ? ahn[r * pH + j - 2 * H] : vi;
        a.dG[((size_t)t * B + row0 + r) * gld + (size_t)(k - a.dg_k0) * GH + j] = vi;
        if (a.dAh) a.dAh[(cell * B + row0 + r) * GH + j] = vh;
        if (a.pdAh_hi) put_plane(a.pdAh_hi, a.pdAh_lo, (cell * B + row0 + r) * GH + j, vh);  // hybrid wavefronts: operand planes
      }
  }
  for (int j = tid; j < GH; j += NT) {
    float s1 = 0.f;
    if (gru && j >= 2 * H) {
      for (int r = 0; r < nrows; ++r) s1 += ahn[r * pH + j - 2 * H];
    } else {
      for (int r = 0; r < nrows; ++r) s1 += S[r * pS + j];
    }
    atomicAdd(&a.g_b_hh[(size_t)k * GH + j], s1);
  }
  if (!gru && t > 0)
    for (int e = tid; e < nrows * H; e += NT) {
      const int r = e / H, j = e - r * H;
      a.dc[(cell * B + row0 + r) * H + j] = ahn[r * pH + j];
    }
  if (!gru && a.single >= 0 && a.dc0_out)
    for (int e = tid; e < nrows * H; e += NT) {
      const int r = e / H, j = e - r * H;
      a.dc0_out[(size_t)(row0 + r) * H + j] = ahn[r * pH + j];
    }

  // ---- I. dh_prev += dA_h @ W_hh ;  J. dz1 += dA_i @ W_ih[:, :Ci] ----------------------------------
  if (!a.skip_hh)  // (hybrid wavefronts: this product is the batched tcgen05 GEMM behind the launch, accumulated into a.dh)
    tile_gemm<RPT, KC>(dact, w.Whh, H, GH, H, sm + sp.wst, [&](int r, int j, float v) { dhr[r * pH + j] += v; },
                   gru ? 2 * H : (1 << 30), gru ? H : 0, 0);
  if (Ci <= 64) skinny_gemm<RPT>(dact, w.WihZ, d.Cip, GH, Ci, sm + sp.wst, [&](int r, int j, float v) { zrow[r * pC + j] += v; });
  else tile_gemm<RPT, KC>(dact, w.WihZ, d.Cip, GH, Ci, sm + sp.wst, [&](int r, int j, float v) { zrow[r * pC + j] += v; });
  __syncthreads();
  if (t > 0)
    for (int e = tid; e < nrows * H; e += NT) {
      const int r = e / H, j = e - r * H;
      a.dh[(cell * B + row0 + r) * H + j] = dhr[r * pH + j];
    }
  if (a.single >= 0 && a.dh0_out)
    for (int e = tid; e < nrows * H; e += NT) {
      const int r = e / H, j = e - r * H;
      a.dh0_out[(size_t)(row0 + r) * H + j] = dhr[r * pH + j];
    }
  for (int e = tid; e < R * C; e += NT) {
    const int r = e / C, c = e - r * C;
    const float v = zrow[r * pC + c];
    zact[c * RS + r] = v;
    if (r < nrows) a.dzf[(cell * B + row0 + r) * C + c] = v;
  }

  // ---- K. dy = dzf @ W^T ; ActNorm backward (modules.py:45-66) --------------------------------------
  tile_gemm<RPT, KC>(zact, w.WT, d.Cp, C, C, sm + sp.wst, [&](int r, int j, float dy) {
    const float y = (r < nrows) ? a.st.y[(cell * B + row0 + r) * C + j] : 0.f;
    dxr[r * pC + j] = dy * expf(w.an_logs[j]);
    prod[r * pO + j] = dy * y;
  });
  __syncthreads();
  if (a.single >= 0) {
    if (a.dx0_out)
      for (int e = tid; e < nrows * C; e += NT) {
        const int r = e / C, c = e - r * C;
        a.dx0_out[(size_t)(row0 + r) * C + c] = dxr[r * pC + c];
      }
  } else if (k > 0) {
    for (int e = tid; e < nrows * C; e += NT) {
      const int r = e / C, c = e - r * C;
      a.dx[(cell * B + row0 + r) * C + c] = dxr[r * pC + c];
    }
  } else if (DXIN) {  // step 0: the gradient of the flow input of frame t (cell == t)
    for (int e = tid; e < nrows * C; e += NT) {
      const int r = e / C, c = e - r * C;
      a.dx_in[(cell * B + row0 + r) * C + c] = dxr[r * pC + c];
    }
  }
  for (int c = tid; c < C; c += NT) {
    float s1 = 0.f, s2 = 0.f;
    for (int r = 0; r < nrows; ++r) { s1 += dxr[r * pC + c]; s2 += prod[r * pO + c]; }
    atomicAdd(&a.g_an_bias[(size_t)k * C + c], s1);
    atomicAdd(&a.g_an_logs[(size_t)k * C + c], s2);
  }
}

template <int RPT, int KC> static int launch_bwd_t(const BwdArgs &a, bool tcw, cudaStream_t st) {  // tcw: hybrid wavefronts
  constexpr int R = Tile<RPT>::R;
  const int bytes = plan_smem(a.d, R, true, false, KC).total * (int)sizeof(float);
  auto kern = a.dx_in ? core_bwd_wave<RPT, KC, true> : core_bwd_wave<RPT, KC, false>;
  LFI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  const int tiles = (a.B + R - 1) / R, K = a.d.K;
  BwdArgs aw = a;
  aw.skip_hh = tcw ? 1 : 0;
  for (int wave = a.Tp + K - 2; wave >= 0; --wave) {
    const int k0 = max(0, wave - a.Tp + 1), k1 = min(K - 1, wave);
    dim3 grid(tiles, k1 - k0 + 1);
    kern<<<grid, NT, bytes, st>>>(aw, wave, k0);
    if (!tcw) continue;
    // cells (k, t = wave - k) with t >= 1 wrote the direct part of d h[k][t-1] into a.dh[k][t]; add dA_h[k][t] W_hh[k]  (batch over k)
    const int kb0 = k0, kb1 = min(k1, wave - 1);
    if (kb1 >= kb0) {
      const int H = a.d.H, GH = a.d.GH, B = a.B, Tp = a.Tp;
      const size_t cell0 = (size_t)kb0 * Tp + (wave - kb0);     // (k, t) of the first cell; next cell: + (Tp - 1)
      GemmArgs q = gemm_args(0, 0, B, H, GH, a.dAh ? a.dAh + cell0 * B * GH : nullptr, GH, nullptr, H, a.dh + cell0 * B * H, H, LFI_EPI_ACCUM);
      q.batch = kb1 - kb0 + 1; q.sA = (long)(Tp - 1) * B * GH; q.sB = (long)GH * H; q.sC = (long)(Tp - 1) * B * H;
      if (a.pdAh_hi)
        q.pA = plane_ref((const uint16_t *)a.pdAh_hi + cell0 * B * GH, a.pdAh_lo ? (const uint16_t *)a.pdAh_lo + cell0 * B * GH : nullptr, GH, q.sA);
      q.pB = plane_ref((const uint16_t *)a.wtc.whh_hi + (size_t)kb0 * GH * H,
                       a.wtc.whh_lo ? (const uint16_t *)a.wtc.whh_lo + (size_t)kb0 * GH * H : nullptr, H, (long)GH * H);
      LFI_TRY(gemm_dispatch(a.wtc.mode, q, a.wtc.gws, a.wtc.gws_bytes, st));
    }
  }
  LFI_LAUNCH_CHECK_N(a.Tp + K - 1);
  return LFI_OK;
}

template <int RPT, int KC> static int launch_bwd_single_t(const BwdArgs &a, cudaStream_t st) {
  constexpr int R = Tile<RPT>::R;
  const int bytes = plan_smem(a.d, R, true, false, KC).total * (int)sizeof(float);
  LFI_CUDA(cudaFuncSetAttribute(core_bwd_wave<RPT, KC, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  core_bwd_wave<RPT, KC, false><<<dim3((a.B + R - 1) / R, 1), NT, bytes, st>>>(a, a.single, a.single);  // wave = k: t = 0
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

int launch_bwd_single(const BwdArgs &a, cudaStream_t st) {
  LFI_REQUIRE(a.single >= 0 && a.single < a.d.K && a.Tp == 1 && a.dz_ext, LFI_ERR_ARG, "flow core backward (single cell): bad arguments");
  int kc = KC16;
  const int rpt = choose_tile(a.d, a.B, true, false, &kc);
  switch (rpt * 100 + kc) {
    case 816: return launch_bwd_single_t<8, 16>(a, st);
    case 416: return launch_bwd_single_t<4, 16>(a, st);
    case 216: return launch_bwd_single_t<2, 16>(a, st);
    case 116: return launch_bwd_single_t<1, 16>(a, st);
    case 808: return launch_bwd_single_t<8, 8>(a, st);
    case 408: return launch_bwd_single_t<4, 8>(a, st);
    case 208: return launch_bwd_single_t<2, 8>(a, st);
    case 108: return launch_bwd_single_t<1, 8>(a, st);
  }
  set_error("flow core backward: shape does not fit shared memory (H=%d G=%d C=%d)", a.d.H, a.d.G, a.d.C);
  return LFI_ERR_SHAPE;
}

static int launch_bwd_wave(const BwdArgs &a, bool tcw, cudaStream_t st) {
  int kc = KC16;
  const int rpt = choose_tile(a.d, a.B, true, false, &kc);
  switch (rpt * 100 + kc) {
    case 816: return launch_bwd_t<8, 16>(a, tcw, st);
    case 416: return launch_bwd_t<4, 16>(a, tcw, st);
    case 216: return launch_bwd_t<2, 16>(a, tcw, st);
    case 116: return launch_bwd_t<1, 16>(a, tcw, st);
    case 808: return launch_bwd_t<8, 8>(a, tcw, st);
    case 408: return launch_bwd_t<4, 8>(a, tcw, st);
    case 208: return launch_bwd_t<2, 8>(a, tcw, st);
    case 108: return launch_bwd_t<1, 8>(a, tcw, st);
  }
  set_error("flow core backward: shape does not fit shared memory (H=%d G=%d C=%d)", a.d.H, a.d.G, a.d.C);
  return LFI_ERR_SHAPE;
}

int launch_bwd(const BwdArgs &a, CoreKernel kern, cudaStream_t st) {
  switch (kern) {
    case CoreKernel::Wave: return launch_bwd_wave(a, false, st);
    case CoreKernel::WaveHybrid:
      LFI_REQUIRE(a.single < 0 && a.wtc.mode && a.wtc.whh_hi, LFI_ERR_ARG, "flow core backward: hybrid wavefronts need W_hh planes");
      return launch_bwd_wave(a, true, st);
    case CoreKernel::Pipe: return launch_bwd_pipe(a, st);
    case CoreKernel::PipeTc: return launch_bwd_pipe_tc(a, st);
  }
  set_error("flow core backward: unknown kernel %d", (int)kern);
  return LFI_ERR_ARG;
}

}  // namespace core
}  // namespace lfi
