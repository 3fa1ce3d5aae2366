// Sequential flow core, forward direction (training / eval) and inverse direction (sampling / invert).
//
//   forward : FlowStep.normal_flow  (models.py:311-342) for every (step k, frame t) cell, scheduled as
//             anti-diagonal wavefronts: cells with k + t = const are independent (cell (k,t) needs the
//             output of (k-1,t) and the RNN state of (k,t-1)), so one launch evaluates up to K cells for
//             all sequence tiles at once.  Weights stream from L2 once per CTA per launch.
//   inverse : FlowStep.reverse_flow (models.py:345-373); strictly serial in (t, k) for a sequence, so one
//             persistent CTA per sequence tile walks all frames and steps with no host round-trip
//             (SeqGlow.inference models.py:581-594 / SeqGlow.invert 617-645).
#include "core_tile.cuh"
#include "core_api.cuh"
#include "core_pipe.cuh"
#include <cstdlib>

namespace lfi {
namespace core {

// ------------------------------------------------------------------------------------------------
// coupling network f_seq (models.py:204-214): S <- gate pre-activations, h (c) update, o = LinearZeros(h)
// in : sm[zact] rows [0,Ci) = z1 (act layout), sm[hp] = h_prev, sm[cp] = c_prev (LSTM)
//      Grow != nullptr: S = G[row] (+ z1 part + h part);  else S already holds b_ih + c @ W_ih[:, Ci:]^T
// out: sm[hp] = h_new, sm[cp] = c_new, sm[orow] = o; optional stashes
template <int RPT, int KC = KC16>
__device__ __forceinline__ void coupling_net(const Dims &d, const StepWeights &w, const SmemPlan &sp, float *sm,
                                             int nrows, const float *Grow, long g_ld, float *st_gates, float *st_ahn,
                                             float *st_h, float *st_c, float *st_o, bool hh_pre = false, const float *gh_rows = nullptr) {
  constexpr int R = Tile<RPT>::R, RS = Tile<RPT>::RS;
  const int tid = threadIdx.x;
  const int H = d.H, GH = d.GH, pS = odd(GH), pH = odd(H), pO = odd(d.Co > d.C ? d.Co : d.C);
  float *S = sm + sp.S, *ahn = sm + sp.ahn, *hp = sm + sp.hp, *cp = sm + sp.cp, *orow = sm + sp.orow;

  // time-parallel part of the gate pre-activations (and, hybrid wavefronts, the recurrent product that came from the batched
  // tcgen05 GEMM; gh_rows == nullptr: zero state, t = 0): requested up front, four rows in flight per thread, so that their
  // DRAM latency is paid once and overlaps the weight stream of the z1 product
  const bool gru = d.G == 3;
  if (Grow) {
    constexpr int NR = R >= 8 ? 8 : 4;  // rows in flight per thread
    for (int r0 = 0; r0 < R; r0 += NR)
      for (int j = tid; j < GH; j += NT) {
        float g[NR], hh[NR];
#pragma unroll
        for (int i = 0; i < NR; ++i) {
          const bool ok = r0 + i < nrows;
          g[i] = ok ? __ldg(Grow + (size_t)(r0 + i) * g_ld + j) : 0.f;
          hh[i] = (hh_pre && gh_rows && ok) ? __ldg(gh_rows + (size_t)(r0 + i) * GH + j) : 0.f;
        }
        const float bh = hh_pre ? w.b_hh[j] : 0.f;
#pragma unroll
        for (int i = 0; i < NR; ++i) {
          if (hh_pre && gru && j >= 2 * H) { ahn[(r0 + i) * pH + (j - 2 * H)] = hh[i] + bh; S[(r0 + i) * pS + j] = g[i]; }
          else S[(r0 + i) * pS + j] = g[i] + hh[i] + bh;
        }
      }
  } else if (hh_pre) {
    __syncthreads();
    for (int r = 0; r < R; ++r)
      for (int j = tid; j < GH; j += NT) {
        float v = w.b_hh[j];
        if (gh_rows && r < nrows) v += gh_rows[(size_t)r * GH + j];
        if (gru && j >= 2 * H) ahn[r * pH + (j - 2 * H)] = v;
        else S[r * pS + j] += v;
      }
  }
  // z1 part
  tile_gemm<RPT, KC>(sm + sp.zact, w.WzT, GH, d.Ci, GH, sm + sp.wst, [&](int r, int j, float v) { S[r * pS + j] += v; });
  // h part
  if (!hh_pre) {
    tile_gemm<RPT, KC>(hp, w.WhhT, GH, H, GH, sm + sp.wst, [&](int r, int j, float v) {
      v += w.b_hh[j];
      if (gru && j >= 2 * H) ahn[r * pH + (j - 2 * H)] = v;
      else S[r * pS + j] += v;
    });
  }
  __syncthreads();
  // gate math: lanes along rows
  for (int e = tid; e < R * H; e += NT) {
    const int r = e % R, m = e / R;
    float *s = S + r * pS;
    if (gru) {
      const float rg = sigmoidf_(s[m]), ug = sigmoidf_(s[H + m]);
      const float ng = tanhf(s[2 * H + m] + rg * ahn[r * pH + m]);
      const float hprev = hp[m * RS + r];
      s[m] = rg; s[H + m] = ug; s[2 * H + m] = ng;
      hp[m * RS + r] = ng + ug * (hprev - ng);
    } else {
      const float ig = sigmoidf_(s[m]), fg = sigmoidf_(s[H + m]), gg = tanhf(s[2 * H + m]), og = sigmoidf_(s[3 * H + m]);
      const float cn = fg * cp[m * RS + r] + ig * gg;
      s[m] = ig; s[H + m] = fg; s[2 * H + m] = gg; s[3 * H + m] = og;
      cp[m * RS + r] = cn;
      hp[m * RS + r] = og * tanhf(cn);
    }
  }
  __syncthreads();
  // stash (coalesced along columns)
  if (st_gates)
    for (int r = 0; r < nrows; ++r)
      for (int j = tid; j < GH; j += NT) st_gates[(size_t)r * GH + j] = S[r * pS + j];
  if (st_ahn && gru)
    for (int r = 0; r < nrows; ++r)
      for (int j = tid; j < H; j += NT) st_ahn[(size_t)r * H + j] = ahn[r * pH + j];
  if (st_h)
    for (int r = 0; r < nrows; ++r)
      for (int j = tid; j < H; j += NT) st_h[(size_t)r * H + j] = hp[j * RS + r];
  if (st_c && !gru)
    for (int r = 0; r < nrows; ++r)
      for (int j = tid; j < H; j += NT) st_c[(size_t)r * H + j] = cp[j * RS + r];
  // LinearZeros (modules.py:93-95)
  if (d.Co <= 64)
    skinny_gemm<RPT>(hp, w.WfT, d.Cop, H, d.Co, sm + sp.wst, [&](int r, int j, float v) {
      orow[r * pO + j] = (v + w.bf[j]) * expf(3.0f * w.lf[j]);
    });
  else
    tile_gemm<RPT, KC>(hp, w.WfT, d.Cop, H, d.Co, sm + sp.wst, [&](int r, int j, float v) {
      orow[r * pO + j] = (v + w.bf[j]) * expf(3.0f * w.lf[j]);
    });
  __syncthreads();
  if (st_o)
    for (int e = tid; e < nrows * d.Co; e += NT) { const int r = e / d.Co, j = e - r * d.Co; st_o[(size_t)r * d.Co + j] = orow[r * pO + j]; }
}

// ------------------------------------------------------------------------------------------------
template <int RPT, int KC>
__global__ void __launch_bounds__(NT) core_fwd_wave(FwdArgs a, int wave, int kmin) {
  extern __shared__ __align__(16) float sm[];
  constexpr int R = Tile<RPT>::R, RS = Tile<RPT>::RS;
  const Dims &d = a.d;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int k = kmin + blockIdx.y, t = wave - k;
  const int row0 = blockIdx.x * R, nrows = min(R, a.B - row0);
  const int C = d.C, Ci = d.Ci, Cz = d.Cz, H = d.H, B = a.B;
  const SmemPlan sp = plan_smem(d, R, false, false, KC);
  const StepWeights w = a.dv.step(d, k);
  const size_t cell = (size_t)k * a.Tp + t;
  const int pC = odd(C), pO = odd(d.Co > C ? d.Co : C);
  float *xs = sm + sp.xs, *zact = sm + sp.zact, *zrow = sm + sp.zrow, *hp = sm + sp.hp, *cp = sm + sp.cp;

  // 1. ActNorm (modules.py:45-66): y = (x + bias) * exp(logs)
  for (int e = tid; e < R * C; e += NT) {
    const int r = e / C, c = e - r * C;
    float v = 0.f;
    if (r < nrows) {
      const int b = row0 + r;
      const float x = (k == a.k_first) ? a.x0[(size_t)b * a.x_sb + (size_t)t * a.x_st + c]
                                       : a.xin[(cell * B + b) * C + c];
      v = (x + w.an_bias[c]) * expf(w.an_logs[c]);
      if (a.st_y) a.st_y[(cell * B + b) * C + c] = v;
    }
    xs[c * RS + r] = v;
  }
  {  // state the cell starts from (four rows requested per thread before the first is used)
    const float *hsrc = t > 0 ? a.st_h + (cell - 1) * B * H : (a.h0 ? a.h0 + (size_t)k * B * H : nullptr);
    const float *csrc = d.G != 4 ? nullptr : (t > 0 ? a.st_c + (cell - 1) * B * H : (a.c0 ? a.c0 + (size_t)k * B * H : nullptr));
    for (int r0 = 0; r0 < R; r0 += 4)
      for (int m = tid; m < H; m += NT) {
        float hv[4], cv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const bool ok = r0 + i < nrows;
          hv[i] = (ok && hsrc) ? hsrc[(size_t)(row0 + r0 + i) * H + m] : 0.f;
          cv[i] = (ok && csrc) ? csrc[(size_t)(row0 + r0 + i) * H + m] : 0.f;
        }
        *reinterpret_cast<float4 *>(hp + m * RS + r0) = make_float4(hv[0], hv[1], hv[2], hv[3]);
        if (d.G == 4) *reinterpret_cast<float4 *>(cp + m * RS + r0) = make_float4(cv[0], cv[1], cv[2], cv[3]);
      }
  }
  // 2. invertible 1x1 conv (modules.py:186): z = y @ W
  tile_gemm<RPT, KC>(xs, w.Wfwd, d.Cp, C, C, sm + sp.wst, [&](int r, int j, float v) {
    zrow[r * pC + j] = v;
    if (j < Ci) zact[j * RS + r] = v;
  });
  __syncthreads();
  if (a.st_zf)
    for (int e = tid; e < nrows * C; e += NT) { const int r = e / C, j = e - r * C; a.st_zf[(cell * B + row0 + r) * C + j] = zrow[r * pC + j]; }

  // 3. coupling network
  const size_t rowbase = cell * B + row0;
  coupling_net<RPT, KC>(d, w, sp, sm, nrows, a.G + ((size_t)t * B + row0) * a.g_ld + (size_t)(k - a.g_k0) * d.GH, a.g_ld,
                    a.st_gates ? a.st_gates + rowbase * d.GH : nullptr, a.st_ahn ? a.st_ahn + rowbase * H : nullptr,
                    a.st_h + rowbase * H, a.st_c ? a.st_c + rowbase * H : nullptr,
                    a.st_o ? a.st_o + rowbase * d.Co : nullptr, a.gh_pre != nullptr,
                    (a.gh_pre && t > 0) ? a.gh_pre + ((size_t)k * B + row0) * d.GH : nullptr);

  if (a.ph_hi)  // hybrid wavefronts: the new state also as the operand plane(s) of the next wavefront's recurrent GEMM (and of dW_hh)
    for (int r = 0; r < nrows; ++r)
      for (int j = tid; j < H; j += NT) put_plane(a.ph_hi, a.ph_lo, (rowbase + r) * H + j, hp[j * RS + r]);

  // 4. coupling (models.py:331-341), log-det, NLL on the last step (modules.py:207-212, models.py:563-565)
  const float *orow = sm + sp.orow;
  const bool last = (k == a.k_last);
  for (int r = warp; r < nrows; r += NT / 32) {
    const int b = row0 + r;
    float lsum = 0.f;
    for (int q = lane; q < Cz; q += 32) {
      const float z2 = zrow[r * pC + Ci + q];
      if (d.affine) {
        const float shift = orow[r * pO + 2 * q], sc = orow[r * pO + 2 * q + 1];
        const float s = fmaxf(sigmoidf_(sc + 2.0f), d.eps);
        zrow[r * pC + Ci + q] = (z2 + shift) * s;
        lsum += logf(s);
        if (a.scale_out) a.scale_out[((size_t)k * B + b) * Cz + q] = s;
      } else {
        zrow[r * pC + Ci + q] = z2 + orow[r * pO + q];
      }
    }
    lsum = warp_sum(lsum);
    __syncwarp();
    float ld = lsum;
    if (k != a.k_first || a.ld_accumulate) ld += a.ld[(size_t)t * B + b];
    if (last && a.nll) {
      float zsq = 0.f;
      for (int c = lane; c < C; c += 32) { const float z = zrow[r * pC + c]; zsq += z * z; }
      zsq = warp_sum(zsq);
      if (lane == 0) a.nll[(size_t)t * B + b] = -(ld - 0.5f * (zsq + (float)C * kLog2Pi)) / kLn2;
    }
    if (lane == 0) a.ld[(size_t)t * B + b] = ld;
  }
  __syncthreads();
  float *dst = last ? a.z_out + (size_t)t * B * C : a.xin + (cell + a.Tp) * B * C;  // XIN[k+1][t]
  for (int e = tid; e < nrows * C; e += NT) { const int r = e / C, j = e - r * C; dst[(size_t)(row0 + r) * C + j] = zrow[r * pC + j]; }
}

// ------------------------------------------------------------------------------------------------
// Persistent inverse kernel: one CTA per sequence tile, all frames of a chunk x all K steps.
// STASH: also store the activations of the step (InvArgs.st_x1 ...; one frame, one step); the instantiation without it is the
// plain inverse
template <int RPT, bool STASH>
__global__ void __launch_bounds__(NT) core_inv_persistent(InvArgs a) {
  extern __shared__ __align__(16) float sm[];
  constexpr int R = Tile<RPT>::R, RS = Tile<RPT>::RS;
  const Dims &d = a.d;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int row0 = blockIdx.x * R, nrows = min(R, a.B - row0);
  const int C = d.C, Ci = d.Ci, Cz = d.Cz, H = d.H, B = a.B, GH = d.GH, D = d.D;
  const bool ar = a.cstatic != nullptr;
  const SmemPlan sp = plan_smem(d, R, false, ar);
  const int pC = odd(C), pO = odd(d.Co > C ? d.Co : C), pS = odd(GH);
  float *xs = sm + sp.xs, *zact = sm + sp.zact, *zrow = sm + sp.zrow, *hp = sm + sp.hp, *cp = sm + sp.cp;
  float *S = sm + sp.S, *cact = sm + sp.cact, *hist = sm + sp.hist, *ldacc = sm + sp.ldacc;
  const int hist0 = d.Far / C;  // p1_face history length

  // AR window (models.py:602): ring of hist0 frame slots; slot `head` holds the oldest frame.
  int head = 0;
  if (ar) {
    for (int e = tid; e < R * d.Far; e += NT) {
      const int r = e / d.Far, i = e - r * d.Far;
      const int s = i / C, c = i - s * C;
      float v = 0.f;
      if (r < nrows) v = a.faces[(size_t)(row0 + r) * a.f_sb + (size_t)(a.t_abs0 - hist0 + s) * a.f_st + c];
      hist[i * RS + r] = v;
    }
  }
  __syncthreads();

  for (int tc = 0; tc < a.Tc; ++tc) {
    // latent for this frame (GaussianDiag.sample output, models.py:511) or the given z (invert)
    for (int e = tid; e < R * C; e += NT) {
      const int r = e / C, c = e - r * C;
      float v = 0.f;
      if (r < nrows && a.noise) v = a.noise[((size_t)(a.t_rel0 + tc) * B + row0 + r) * C + c];
      zrow[r * pC + c] = v;
      if (c < Ci) zact[c * RS + r] = v;
    }
    if (tid < R) ldacc[tid] = 0.f;
    __syncthreads();
    for (int k = a.k_hi; k >= a.k_lo; --k) {
      const StepWeights w = a.dv.step(d, k);
      for (int e = tid; e < R * H; e += NT) {
        const int r = e / H, m = e - r * H;
        float hv = 0.f, cv = 0.f;
        if (r < nrows) {
          hv = a.hstate[((size_t)k * B + row0 + r) * H + m];
          if (d.G == 4) cv = a.cstate[((size_t)k * B + row0 + r) * H + m];
        }
        hp[m * RS + r] = hv;
        if (d.G == 4) cp[m * RS + r] = cv;
      }
      const float *Grow = nullptr;
      if (ar) {
        // cond_transform (models.py:187-190) = static columns (precomputed, incl. bias) + autoregressive
        // p1_face window columns; then the c-part of the gate-ih product.
        const float *cs = a.cstatic + ((size_t)tc * B + row0) * a.cs_ld + (size_t)k * D;
        tile_gemm<RPT>(hist, w.WcArT, D, d.Far, D, sm + sp.wst, [&](int r, int j, float v) {
          v += (r < nrows) ? cs[(size_t)r * a.cs_ld + j] : 0.f;
          cact[j * RS + r] = v > 0.f ? v : kLeaky * v;
        }, (hist0 - head) * C, head * C - d.Far, head * C);
        tile_gemm<RPT>(cact, w.WihCT, GH, D, GH, sm + sp.wst, [&](int r, int j, float v) { S[r * pS + j] = v + w.b_ih[j]; });
      } else {
        Grow = a.G + ((size_t)tc * B + row0) * a.g_ld + (size_t)(k - a.g_k0) * GH;
      }
      coupling_net<RPT>(d, w, sp, sm, nrows, Grow, a.g_ld, STASH ? a.st_gates + (size_t)row0 * GH : nullptr,
                        STASH && a.st_ahn ? a.st_ahn + (size_t)row0 * H : nullptr,
                        a.hstate + ((size_t)k * B + row0) * H, d.G == 4 ? a.cstate + ((size_t)k * B + row0) * H : nullptr,
                        STASH ? a.st_o + (size_t)row0 * d.Co : nullptr);
      // inverse coupling (models.py:358-366): z2 = z2 / scale - shift
      const float *orow = sm + sp.orow;
      for (int r = warp; r < R; r += NT / 32) {
        float lsum = 0.f;
        for (int q = lane; q < Cz; q += 32) {
          const float z2 = zrow[r * pC + Ci + q];
          float v;
          if (d.affine) {
            const float shift = orow[r * pO + 2 * q], sc = orow[r * pO + 2 * q + 1];
            const float s = fmaxf(sigmoidf_(sc + 2.0f), d.eps);
            v = z2 / s - shift;
            lsum += logf(s);
          } else {
            v = z2 - orow[r * pO + q];
          }
          xs[(Ci + q) * RS + r] = v;
        }
        for (int c = lane; c < Ci; c += 32) xs[c * RS + r] = zrow[r * pC + c];
        lsum = warp_sum(lsum);
        if (lane == 0) ldacc[r] -= lsum;
      }
      // 1x1 conv inverse then ActNorm inverse (modules.py:175-177, 189-193, 76-78)
      tile_gemm<RPT>(xs, w.Winv, d.Cp, C, C, sm + sp.wst, [&](int r, int j, float v) {
        if (STASH && r < nrows) {  // xs = zc is complete and unchanged while the product runs ([B][C] of one step: int offsets)
          const int o = (row0 + r) * C + j;
          a.st_zc[o] = xs[j * RS + r];
          a.st_x1[o] = v;
        }
        const float x = v * expf(-w.an_logs[j]) - w.an_bias[j];
        zrow[r * pC + j] = x;
        if (j < Ci) zact[j * RS + r] = x;
      });
      __syncthreads();
    }
    // emit the frame, slide the autoregressive window
    const int t_abs = a.t_abs0 + tc;
    for (int e = tid; e < nrows * C; e += NT) {
      const int r = e / C, c = e - r * C;
      a.faces_out[(size_t)(row0 + r) * a.fo_sb + (size_t)t_abs * a.fo_st + c] = zrow[r * pC + c];
    }
    if (a.logdet_out && tid < nrows) a.logdet_out[(size_t)(a.t_rel0 + tc) * B + row0 + tid] = ldacc[tid];
    if (ar) {
      for (int e = tid; e < R * C; e += NT) {
        const int r = e / C, c = e - r * C;
        hist[(head * C + c) * RS + r] = zrow[r * pC + c];
      }
      head = (head + 1) % hist0;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// host side

constexpr int kMaxSmem = 227 * 1024;

int fwd_smem_bytes(const Dims &d, int R) { return plan_smem(d, R, false, false).total * (int)sizeof(float); }

// Rows per CTA = 4*RPT.  Larger tiles amortise the weight stream, smaller tiles expose more CTAs;
// take the largest tile that still gives every SM a CTA.  The wavefront cell kernels
// may also halve the weight ring (kc = 8) when that is what lets a tile fit (wide shapes: H = 256, LSTM).
int choose_tile(const Dims &d, int B, bool bwd, bool sampler, int *kc_out) {
  const int cand[4] = {8, 4, 2, 1};
  int best = 0, best_kc = KC16;
  for (int i = 0; i < 4; ++i) {
    const int rpt = cand[i], R = RG * rpt;
    int kc = KC16;
    if (plan_smem(d, R, bwd, sampler, kc).total * (int)sizeof(float) > kMaxSmem) {
      kc = 8;
      if (sampler || !kc_out || plan_smem(d, R, bwd, sampler, kc).total * (int)sizeof(float) > kMaxSmem) continue;
    }
    const long ctas = (long)((B + R - 1) / R) * (sampler ? 1 : d.K);
    best = rpt; best_kc = kc;
    if (ctas >= (sampler ? 120 : 148)) break;
  }
  if (kc_out) *kc_out = best_kc;
  return best;  // smallest tile that fits (0 = nothing fits)
}

int choose_rpt(const Dims &d, int B, bool bwd, bool sampler) { return choose_tile(d, B, bwd, sampler, nullptr); }

template <int RPT, int KC> static int launch_fwd_t(const FwdArgs &a, bool tcw, cudaStream_t st) {  // tcw: hybrid wavefronts
  constexpr int R = Tile<RPT>::R;
  const int bytes = plan_smem(a.d, R, false, false, KC).total * (int)sizeof(float);
  LFI_CUDA(cudaFuncSetAttribute(core_fwd_wave<RPT, KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  const int tiles = (a.B + R - 1) / R;
  const int nk = a.k_last - a.k_first + 1;
  for (int wave = 0; wave < a.Tp + nk - 1; ++wave) {
    // active steps: k_first + i with 0 <= wave - i < Tp
    const int i0 = max(0, wave - a.Tp + 1), i1 = min(nk - 1, wave);
    dim3 grid(tiles, i1 - i0 + 1);
    if (!tcw) {
      core_fwd_wave<RPT, KC><<<grid, NT, bytes, st>>>(a, wave + a.k_first, a.k_first + i0);
      continue;
    }
    FwdArgs aw = a;
    float *gh = a.wtc.ghbuf + (size_t)(wave & 1) * a.d.K * a.B * a.d.GH;
    aw.gh_pre = gh;
    // cells (k, t = wave - k) with t >= 1: k in [i0, min(i1, wave - 1)];  gh[k] = h[k][t-1] W_hh[k]^T   (batch over k)
    const int kb0 = i0, kb1 = min(i1, wave - 1);
    if (kb1 >= kb0) {
      const int H = a.d.H, GH = a.d.GH, B = a.B, Tp = a.Tp;
      const size_t cellA = (size_t)kb0 * Tp + (wave - kb0 - 1);   // (k, t-1) of the first cell; next cell: + (Tp - 1)
      GemmArgs q = gemm_args(0, 1, B, GH, H, a.st_h + cellA * B * H, H, nullptr, H, gh + (size_t)kb0 * B * GH, GH, 0);
      q.batch = kb1 - kb0 + 1; q.sA = (long)(Tp - 1) * B * H; q.sB = (long)GH * H; q.sC = (long)B * GH;
      if (a.ph_hi)  // the cells wrote their state as operand planes: no split pass in front of the product
        q.pA = plane_ref((const uint16_t *)a.ph_hi + cellA * B * H, a.ph_lo ? (const uint16_t *)a.ph_lo + cellA * B * H : nullptr, H, q.sA);
      q.pB = plane_ref((const uint16_t *)a.wtc.whh_hi + (size_t)kb0 * GH * H,
                       a.wtc.whh_lo ? (const uint16_t *)a.wtc.whh_lo + (size_t)kb0 * GH * H : nullptr, H, (long)GH * H);
      LFI_TRY(gemm_dispatch(a.wtc.mode, q, a.wtc.gws, a.wtc.gws_bytes, st));
    }
    core_fwd_wave<RPT, KC><<<grid, NT, bytes, st>>>(aw, wave, i0);
  }
  LFI_LAUNCH_CHECK_N(a.Tp + nk - 1);
  return LFI_OK;
}

static int launch_fwd_wave(const FwdArgs &a, bool tcw, cudaStream_t st) {
  int kc = KC16;
  const int rpt = choose_tile(a.d, a.B, false, false, &kc);
  switch (rpt * 100 + kc) {
    case 816: return launch_fwd_t<8, 16>(a, tcw, st);
    case 416: return launch_fwd_t<4, 16>(a, tcw, st);
    case 216: return launch_fwd_t<2, 16>(a, tcw, st);
    case 116: return launch_fwd_t<1, 16>(a, tcw, st);
    case 808: return launch_fwd_t<8, 8>(a, tcw, st);
    case 408: return launch_fwd_t<4, 8>(a, tcw, st);
    case 208: return launch_fwd_t<2, 8>(a, tcw, st);
    case 108: return launch_fwd_t<1, 8>(a, tcw, st);
  }
  set_error("flow core: shape does not fit shared memory (H=%d G=%d C=%d)", a.d.H, a.d.G, a.d.C);
  return LFI_ERR_SHAPE;
}

int launch_fwd(const FwdArgs &a, CoreKernel kern, cudaStream_t st) {
  // Initial state: the plain wavefronts read h0 / c0 (module API, time-chunked evaluation; the caller takes the final state
  // from st_h / st_c).  The stage pipelines (GRU only) run their carry instantiation when given h0 and h_last.  The hybrid
  // wavefronts start from zeros: their batched recurrent product would need h0 as operand planes.
  switch (kern) {
    case CoreKernel::Wave:
      LFI_REQUIRE(!a.h_last, LFI_ERR_ARG, "flow core: the wavefront kernels do not write h_last");
      return launch_fwd_wave(a, false, st);
    case CoreKernel::WaveHybrid:
      LFI_REQUIRE(!a.h0 && !a.c0 && !a.h_last, LFI_ERR_ARG, "flow core: the hybrid wavefronts take no initial state");
      LFI_REQUIRE(a.k_first == 0 && a.wtc.mode && a.wtc.whh_hi && a.wtc.ghbuf, LFI_ERR_ARG,
                  "flow core: hybrid wavefronts need W_hh planes and product buffers from step 0");
      return launch_fwd_wave(a, true, st);
    case CoreKernel::Pipe:
      LFI_REQUIRE(!a.c0, LFI_ERR_ARG, "flow core: the stage pipelines carry no LSTM cell state");
      return launch_fwd_pipe(a, st);
    case CoreKernel::PipeTc:
      LFI_REQUIRE(!a.c0, LFI_ERR_ARG, "flow core: the stage pipelines carry no LSTM cell state");
      return launch_fwd_pipe_tc(a, st);
  }
  set_error("flow core: unknown kernel %d", (int)kern);
  return LFI_ERR_ARG;
}

template <int RPT> static int launch_inv_t(const InvArgs &a, cudaStream_t st) {
  constexpr int R = Tile<RPT>::R;
  const int bytes = plan_smem(a.d, R, false, a.cstatic != nullptr).total * (int)sizeof(float);
  auto kern = a.st_x1 ? core_inv_persistent<RPT, true> : core_inv_persistent<RPT, false>;
  LFI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  kern<<<(a.B + R - 1) / R, NT, bytes, st>>>(a);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

int launch_inv(const InvArgs &a, cudaStream_t st) {
  if (use_inv_rows(a)) return launch_inv_rows(a, st);
  const int rpt = choose_rpt(a.d, a.B, false, true);
  switch (rpt) {
    case 8: return launch_inv_t<8>(a, st);
    case 4: return launch_inv_t<4>(a, st);
    case 2: return launch_inv_t<2>(a, st);
    case 1: return launch_inv_t<1>(a, st);
  }
  set_error("flow sampler: shape does not fit shared memory (H=%d D=%d C=%d)", a.d.H, a.d.D, a.d.C);
  return LFI_ERR_SHAPE;
}

}  // namespace core
}  // namespace lfi
