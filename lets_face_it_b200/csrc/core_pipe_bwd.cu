// Persistent stage-pipelined flow core, backward direction (see core_pipe.cuh for the scheme).
//
// Stage k (one 2-CTA cluster) walks the frames in reverse; cell (k, t) consumes d(output of step k) published by
// stage k+1 and the state gradient d h[k][t] it carries itself across frames (registers + one exchange buffer),
// and publishes d(input of step k) to stage k-1.  Each CTA owns 64 hidden units: its 192 gate columns of W_hh /
// W_ih[:, :Ci] are resident in shared memory as [gate column][.] so that dh_prev = dA_h W_hh and dz1 = dA_i W_ih
// are reductions over the CTA's own gate gradients; the partial sums that belong to the other CTA (its hidden
// units / its rows) travel through distributed shared memory.  Per-channel parameter gradients are accumulated in
// registers over all frames and flushed with one round of atomics at the end of the launch.
#include "core_pipe.cuh"
#include <cooperative_groups.h>
#include <cstdlib>

namespace cg = cooperative_groups;

namespace lfi {
namespace core {

__device__ __forceinline__ void st_release_gpu_b(int *p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}

struct PipePlanB {  // offsets in floats
  int whh, wz, wf, wT, vec, dact, dhc, dzf, dor, dz1, total;
  int pC, pO;
};
constexpr int PZ1 = 32;
__device__ int g_core_timing_b = 0;  // debug: LFI_CORE_TIMING=1 prints the phase cycle counts of one CTA  // row pitch of the dz1 partial-sum buffers (Cip <= 32)

__host__ __device__ inline PipePlanB plan_pipe_bwd(const Dims &d) {
  PipePlanB p;
  int o = 0;
  auto take = [&](int n) { int r = o; o += round_up(n, 4); return r; };
  p.pC = odd(d.C);
  p.pO = odd(d.Co);
  p.whh = take(3 * PUC * d.H);      // [g*64 + u][m]      = W_hh[g*H + 64c + u][m]
  p.wz = take(3 * PUC * d.Cip);     // [g*64 + u][i]      = W_ih[g*H + 64c + u][i], i < Ci
  p.wf = take(d.Co * PUC);          // [j][u]             = Wf[j][64c + u]
  p.wT = take(d.C * d.Cp);          // [i][j]             = W[j][i]
  p.vec = take(d.C + d.Co);         // exp(an_logs), exp(3 lf)
  p.dact = take(2 * PUC * PHS);     // two staging buffers [64 units][rows]; buffer 1 doubles as dlin [Co][rows]
  p.dhc = take(PUC * PHS);          // peer's partial of dh_prev for this CTA's units
  p.dzf = take(PRH * p.pC);         // row-major d(1x1 conv output) of this CTA's rows
  p.dor = take(PRH * p.pO);         // row-major dlin of this CTA's rows
  p.dz1 = take(2 * PRH * PZ1);      // dz1 partial sums of this CTA's rows, one slot per producing CTA
  p.total = o;
  return p;
}

// DXIN: stage 0 also stores the gradient of the flow input (BwdArgs.dx_in); the instantiation without it is the plain backward
template <bool DXIN>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(PNT, 1)
core_bwd_pipe(const BwdArgs a, const int P, const int ntiles, int *progress) {
  extern __shared__ __align__(16) float sm[];
  cg::cluster_group cluster = cg::this_cluster();
  const Dims &d = a.d;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = (int)cluster.block_rank();
  const int k = blockIdx.y, K = d.K, p = blockIdx.z;
  const int C = d.C, Ci = d.Ci, Cz = d.Cz, Co = d.Co, H = d.H, GH = d.GH, B = a.B, Tp = a.Tp, Cp = d.Cp, Cip = d.Cip;
  const PipePlanB pl = plan_pipe_bwd(d);
  const int pC = pl.pC, pO = pl.pO;
  float *whh = sm + pl.whh, *wz = sm + pl.wz, *wf = sm + pl.wf, *wT = sm + pl.wT;
  float *ans = sm + pl.vec, *e3 = ans + C;
  float *buf0 = sm + pl.dact, *buf1 = buf0 + PUC * PHS, *dlin = buf1, *dhc = sm + pl.dhc;
  float *dzf = sm + pl.dzf, *dor = sm + pl.dor, *dz1 = sm + pl.dz1;
  float *peer = cluster.map_shared_rank(sm, c ^ 1);
  const StepWeights w = a.dv.step(d, k);
  const bool lastk = (k == K - 1);

  // ---- resident weights -------------------------------------------------------------------------
  for (int e = tid; e < 3 * PUC * (H / 4); e += PNT) {
    const int j = e / (H / 4), m4 = e - j * (H / 4), g = j / PUC, u = j - g * PUC;
    *reinterpret_cast<float4 *>(whh + j * H + 4 * m4) = *reinterpret_cast<const float4 *>(w.Whh + (size_t)(g * H + PUC * c + u) * H + 4 * m4);
  }
  for (int e = tid; e < 3 * PUC * (Cip / 4); e += PNT) {
    const int j = e / (Cip / 4), i4 = e - j * (Cip / 4), g = j / PUC, u = j - g * PUC;
    *reinterpret_cast<float4 *>(wz + j * Cip + 4 * i4) = *reinterpret_cast<const float4 *>(w.WihZ + (size_t)(g * H + PUC * c + u) * Cip + 4 * i4);
  }
  for (int e = tid; e < Co * (PUC / 4); e += PNT) {
    const int j = e / (PUC / 4), u4 = e - j * (PUC / 4);
    *reinterpret_cast<float4 *>(wf + j * PUC + 4 * u4) = *reinterpret_cast<const float4 *>(w.Wf + (size_t)j * H + PUC * c + 4 * u4);
  }
  for (int e = tid; e < C * (Cp / 4); e += PNT)
    *reinterpret_cast<float4 *>(wT + 4 * e) = *reinterpret_cast<const float4 *>(w.WT + 4 * e);
  for (int e = tid; e < C; e += PNT) ans[e] = expf(w.an_logs[e]);
  for (int e = tid; e < Co; e += PNT) e3[e] = expf(3.0f * w.lf[e]);
  cluster.sync();

  const int ul = (warp & 3) * 8 + (lane & 7), rg = (warp >> 2) * 4 + (lane >> 3);
  const int u0 = 2 * ul, uo = PUC * c + u0, up = PUC * (c ^ 1) + u0;
  const int lr0 = PRH * c;
  const int ncq = Cp >> 2, nciq = Cip >> 2;
  const int kcq = tid % ncq, krp = tid / ncq;     // 1x1 conv backward: rows 2krp, 2krp+1 x columns 4kcq..
  const int jcq = tid % nciq, jrp = tid / nciq;   // dz1: tile rows 2jrp, 2jrp+1 x columns 4jcq..
  const bool kact = krp < PRH / 2, jact = jrp < PR / 2;
  const int *wait_flag = progress + ((size_t)(p * K + k + 1) * 2 + c);
  int *my_flag = progress + ((size_t)(p * K + k) * 2 + c);
  int it = 0;
  bool x3_pending = false;
  const bool timing = g_core_timing_b && tid == 0 && c == 0 && p == 0 && (k == 8 || k == 0 || k == K - 1);
  long long tacc[12] = {0}, tprev = 0;
#define TSTAMPB(i) do { if (timing) { const long long now_ = clock64(); tacc[i] += now_ - tprev; tprev = now_; } } while (0)

  // per-channel gradient accumulators (flushed once at the end)
  float gbhh[3][2] = {{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}}, gbin[2] = {0.f, 0.f};
  float gbf[2] = {0.f, 0.f}, glf[2] = {0.f, 0.f};
  float gab[4] = {0.f, 0.f, 0.f, 0.f}, gal[4] = {0.f, 0.f, 0.f, 0.f};

  for (int tile = p; tile < ntiles; tile += P) {
    const int row0 = tile * PR, nrows = min(PR, B - row0);
    const int nmy = max(0, min(PRH, nrows - lr0));
    float carry[8][2];  // d h[k][t] arriving from frame t+1 (this thread's rows x units)
#pragma unroll
    for (int r = 0; r < 8; ++r) carry[r][0] = carry[r][1] = 0.f;

    for (int t = Tp - 1; t >= 0; --t, ++it) {
      const size_t cell = (size_t)k * Tp + t;
      if (timing) tprev = clock64();
      // ---- 0. prefetch the gate stash of this thread's 8 rows x 2 units ----------------------------------------------
      float2 pg[8][3], pa[8], ph[8];
      {
        const size_t rb = cell * B + row0 + 8 * rg;
        if (a.stash_tiled) {  // layout of the tensor-core forward pipeline (core_pipe.cuh: stash_tiled_off)
          const int hs = u0 >> 4, i4 = (u0 & 15) >> 2, eo = (u0 & 3) + 4 * (8 * rg);
          const float *gq = a.st.gates + stash_tiled_off(cell, ntiles, tile, c, hs, 3, 0, i4) + eo;
          const float *aq = a.st.ahn + stash_tiled_off(cell, ntiles, tile, c, hs, 1, 0, i4) + eo;
          const float *hq = a.st.h + stash_tiled_off(cell - (t > 0 ? 1 : 0), ntiles, tile, c, hs, 1, 0, i4) + eo;
#pragma unroll
          for (int r = 0; r < 8; ++r) {
            if (8 * rg + r < nrows) {
              pg[r][0] = __ldg(reinterpret_cast<const float2 *>(gq + 4 * r));
              pg[r][1] = __ldg(reinterpret_cast<const float2 *>(gq + 1024 + 4 * r));
              pg[r][2] = __ldg(reinterpret_cast<const float2 *>(gq + 2048 + 4 * r));
              pa[r] = __ldg(reinterpret_cast<const float2 *>(aq + 4 * r));
              ph[r] = t > 0 ? __ldg(reinterpret_cast<const float2 *>(hq + 4 * r)) : make_float2(0.f, 0.f);
            } else {
              pg[r][0] = pg[r][1] = pg[r][2] = pa[r] = ph[r] = make_float2(0.f, 0.f);
            }
          }
        } else
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          if (8 * rg + r < nrows) {
            const float *gq = a.st.gates + (rb + r) * GH + uo;
            pg[r][0] = __ldg(reinterpret_cast<const float2 *>(gq));
            pg[r][1] = __ldg(reinterpret_cast<const float2 *>(gq + H));
            pg[r][2] = __ldg(reinterpret_cast<const float2 *>(gq + 2 * H));
            pa[r] = __ldg(reinterpret_cast<const float2 *>(a.st.ahn + (rb + r) * H + uo));
            ph[r] = t > 0 ? __ldg(reinterpret_cast<const float2 *>(a.st.h + (rb + r - (size_t)B) * H + uo)) : make_float2(0.f, 0.f);
          } else {
            pg[r][0] = pg[r][1] = pg[r][2] = pa[r] = ph[r] = make_float2(0.f, 0.f);
          }
        }
      }
      float yv[2][4];  // ActNorm outputs of this thread's 1x1-conv-backward outputs (d logs), requested early
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int r = 2 * krp + i;
          yv[i][j] = (kact && r < nmy && 4 * kcq + j < C) ? __ldg(a.st.y + (cell * B + row0 + lr0 + r) * C + 4 * kcq + j) : 0.f;
        }
      // coupling stash of this CTA's rows (lane = coupling channel, row = warp + 8n): independent of stage k+1, requested
      // before the wait so that the latency hides behind it
      constexpr int NR = PRH / 8;
      float c_dnl[NR], c_z2[NR];
      float2 c_o[NR];
#pragma unroll
      for (int n = 0; n < NR; ++n) {
        const int r = warp + 8 * n, q = lane;
        c_dnl[n] = 0.f; c_z2[n] = 0.f; c_o[n] = make_float2(0.f, 0.f);
        if (r < nmy) {
          const int b = row0 + lr0 + r;
          c_dnl[n] = a.dnll[(size_t)t * B + b];
          if (q < Cz) {
            if (d.affine) {
              c_o[n] = *reinterpret_cast<const float2 *>(a.st.o + (cell * B + b) * Co + 2 * q);
              c_z2[n] = a.st.zf[(cell * B + b) * C + Ci + q];
            } else {
              c_o[n].x = a.st.o[(cell * B + b) * Co + q];
            }
          }
        }
      }
      // ---- 1. wait for stage k+1 ---------------------------------------------------------------------------------------
      if (!lastk) {
        if (tid == 0) {
          spin_wait_gt(wait_flag, it);
        }
        __syncthreads();
      }
      TSTAMPB(0);
      // ---- 2. coupling backward (models.py:331-341) on this CTA's 32 rows ---------------------------------------------
      float c_dz[NR], c_dx1[NR];
#pragma unroll
      for (int n = 0; n < NR; ++n) {  // the published d(output of step k): all requests first
        const int r = warp + 8 * n, q = lane;
        c_dz[n] = 0.f; c_dx1[n] = 0.f;
        if (r < nmy) {
          const int b = row0 + lr0 + r;
          const float *dxp = a.dx + ((cell + Tp) * B + b) * C;
          const float *zp = a.z + ((size_t)t * B + b) * C;
          if (q < Cz) c_dz[n] = lastk ? c_dnl[n] * zp[Ci + q] / kLn2 : __ldcg(dxp + Ci + q);  // last step: d nll / d z = z / ln2
          if (q < Ci) c_dx1[n] = lastk ? c_dnl[n] * zp[q] / kLn2 : __ldcg(dxp + q);
        }
      }
#pragma unroll
      for (int n = 0; n < NR; ++n) {
        const int r = warp + 8 * n, q = lane;
        float dz2 = 0.f, dl0 = 0.f, dl1 = 0.f;
        if (r < nmy && q < Cz) {
          const float dld = -c_dnl[n] / kLn2;  // d nll / d logdet
          const float dz2n = c_dz[n];
          if (d.affine) {
            const float shift = c_o[n].x, sc = c_o[n].y, z2 = c_z2[n];
            const float sg = fast_sigmoid(sc + 2.0f), s = fmaxf(sg, d.eps);
            const float ds = dz2n * (z2 + shift) + dld / s;
            dz2 = dz2n * s;
            const float dsc = (sg >= d.eps) ? ds * sg * (1.0f - sg) : 0.f;
            gbf[0] += dz2; gbf[1] += dsc; glf[0] += dz2 * shift; glf[1] += dsc * sc;
            dl0 = dz2 * e3[2 * q]; dl1 = dsc * e3[2 * q + 1];
          } else {
            const float ov = c_o[n].x;
            dz2 = dz2n;
            gbf[0] += dz2n; glf[0] += dz2n * ov;
            dl0 = dz2n * e3[q];
          }
        }
        if (q < Cz) {
          dzf[r * pC + Ci + q] = dz2;
          if (d.affine) { dor[r * pO + 2 * q] = dl0; dor[r * pO + 2 * q + 1] = dl1; }
          else dor[r * pO + q] = dl0;
        }
        if (q < Ci) dzf[r * pC + q] = c_dx1[n];
      }
      __syncthreads();
      if (x3_pending) { asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory"); x3_pending = false; }  // peer done with buffer 1
      for (int e = tid; e < Co * PRH; e += PNT) {  // dlin in act layout, to both CTAs
        const int j = e / PRH, r = e - j * PRH;
        const float v = dor[r * pO + j];
        dlin[j * PHS + lr0 + r] = v;
        peer[pl.dact + PUC * PHS + j * PHS + lr0 + r] = v;
      }
      TSTAMPB(1);
      cluster.sync();  // X1: dlin of all 64 rows present in both CTAs
      TSTAMPB(2);
      if (t < Tp - 1) {
#pragma unroll
        for (int x = 0; x < 2; ++x) {  // the peer's share of d h[k][t] (it rewrites this buffer only after X2 of this frame)
          const float4 v0 = *reinterpret_cast<const float4 *>(dhc + (u0 + x) * PHS + 8 * rg);
          const float4 v1 = *reinterpret_cast<const float4 *>(dhc + (u0 + x) * PHS + 8 * rg + 4);
          carry[0][x] += v0.x; carry[1][x] += v0.y; carry[2][x] += v0.z; carry[3][x] += v0.w;
          carry[4][x] += v1.x; carry[5][x] += v1.y; carry[6][x] += v1.z; carry[7][x] += v1.w;
        }
      }

      // ---- 3. dh = dlin @ Wf (+ carried gradient) for this thread's rows x units ---------------------------------------
      float dh[8][2];
#pragma unroll
      for (int r = 0; r < 8; ++r) { dh[r][0] = carry[r][0]; dh[r][1] = carry[r][1]; }
#pragma unroll 4
      for (int j = 0; j < Co; ++j) {
        const float4 a0 = *reinterpret_cast<const float4 *>(dlin + j * PHS + 8 * rg);
        const float4 a1 = *reinterpret_cast<const float4 *>(dlin + j * PHS + 8 * rg + 4);
        const float2 wv = *reinterpret_cast<const float2 *>(wf + j * PUC + u0);
        const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
        for (int r = 0; r < 8; ++r) { dh[r][0] = fmaf(av[r], wv.x, dh[r][0]); dh[r][1] = fmaf(av[r], wv.y, dh[r][1]); }
      }
      TSTAMPB(3);
      // ---- 4. GRU gate backward ------------------------------------------------------------------------------------------
      float dar[8][2], dau[8][2], dan[8][2], dnr[8][2];
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int x = 0; x < 2; ++x) {
          const float rgt = x ? pg[r][0].y : pg[r][0].x, ug = x ? pg[r][1].y : pg[r][1].x, ng = x ? pg[r][2].y : pg[r][2].x;
          const float an = x ? pa[r].y : pa[r].x, hpv = x ? ph[r].y : ph[r].x;
          const float g = dh[r][x];
          const float dn = g * (1.0f - ug), du = g * (hpv - ng);
          const float v_an = dn * (1.0f - ng * ng);
          dan[r][x] = v_an;
          dau[r][x] = du * ug * (1.0f - ug);
          dar[r][x] = v_an * an * rgt * (1.0f - rgt);
          dnr[r][x] = v_an * rgt;
          carry[r][x] = g * ug;
          gbhh[0][x] += dar[r][x]; gbhh[1][x] += dau[r][x]; gbhh[2][x] += dnr[r][x]; gbin[x] += v_an;
        }
      {  // dA_i -> dG (time-parallel backward), dA_h stash (dW_hh)
        const size_t ldg = (size_t)K * GH;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          if (8 * rg + r < nrows) {
            const int b = row0 + 8 * rg + r;
            const size_t go = ((size_t)t * B + b) * ldg + (size_t)k * GH + uo, ho = (cell * B + b) * GH + uo;
            if (a.dG) {
              float *gq = a.dG + go;
              *reinterpret_cast<float2 *>(gq) = make_float2(dar[r][0], dar[r][1]);
              *reinterpret_cast<float2 *>(gq + H) = make_float2(dau[r][0], dau[r][1]);
              *reinterpret_cast<float2 *>(gq + 2 * H) = make_float2(dan[r][0], dan[r][1]);
            }
            if (a.dAh) {
              float *hq = a.dAh + ho;
              *reinterpret_cast<float2 *>(hq) = make_float2(dar[r][0], dar[r][1]);
              *reinterpret_cast<float2 *>(hq + H) = make_float2(dau[r][0], dau[r][1]);
              *reinterpret_cast<float2 *>(hq + 2 * H) = make_float2(dnr[r][0], dnr[r][1]);
            }
            if (a.pdG_hi) {
              put_plane2(a.pdG_hi, a.pdG_lo, go, dar[r][0], dar[r][1]);
              put_plane2(a.pdG_hi, a.pdG_lo, go + H, dau[r][0], dau[r][1]);
              put_plane2(a.pdG_hi, a.pdG_lo, go + 2 * H, dan[r][0], dan[r][1]);
            }
            if (a.pdAh_hi) {
              put_plane2(a.pdAh_hi, a.pdAh_lo, ho, dar[r][0], dar[r][1]);
              put_plane2(a.pdAh_hi, a.pdAh_lo, ho + H, dau[r][0], dau[r][1]);
              put_plane2(a.pdAh_hi, a.pdAh_lo, ho + 2 * H, dnr[r][0], dnr[r][1]);
            }
          }
        }
      }
      TSTAMPB(4);
      // ---- 5. dh_prev partial = dA_h W_hh (own units -> carry, peer units -> peer) ; dz1 partial = dA_i W_ih[:, :Ci] -----
      float ip[8][4], jp[2][4];
#pragma unroll
      for (int r = 0; r < 8; ++r) ip[r][0] = ip[r][1] = ip[r][2] = ip[r][3] = 0.f;
#pragma unroll
      for (int i = 0; i < 2; ++i) jp[i][0] = jp[i][1] = jp[i][2] = jp[i][3] = 0.f;
      auto stage_to = [&](float *buf, const float (&v)[8][2]) {
#pragma unroll
        for (int x = 0; x < 2; ++x) {
          *reinterpret_cast<float4 *>(buf + (u0 + x) * PHS + 8 * rg) = make_float4(v[0][x], v[1][x], v[2][x], v[3][x]);
          *reinterpret_cast<float4 *>(buf + (u0 + x) * PHS + 8 * rg + 4) = make_float4(v[4][x], v[5][x], v[6][x], v[7][x]);
        }
      };
      auto acc_i = [&](const float *buf, int g) {
        const float *wb = whh + (size_t)(g * PUC) * H;
#pragma unroll 4
        for (int u = 0; u < PUC; ++u) {
          const float4 a0 = *reinterpret_cast<const float4 *>(buf + u * PHS + 8 * rg);
          const float4 a1 = *reinterpret_cast<const float4 *>(buf + u * PHS + 8 * rg + 4);
          const float2 wo = *reinterpret_cast<const float2 *>(wb + u * H + uo);
          const float2 wp = *reinterpret_cast<const float2 *>(wb + u * H + up);
          const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
          for (int r = 0; r < 8; ++r) {
            ip[r][0] = fmaf(av[r], wo.x, ip[r][0]); ip[r][1] = fmaf(av[r], wo.y, ip[r][1]);
            ip[r][2] = fmaf(av[r], wp.x, ip[r][2]); ip[r][3] = fmaf(av[r], wp.y, ip[r][3]);
          }
        }
      };
      auto acc_j = [&](const float *buf, int g) {
        if (!jact) return;
        const float *wb = wz + (size_t)(g * PUC) * Cip + 4 * jcq;
#pragma unroll 4
        for (int u = 0; u < PUC; ++u) {
          const float2 av = *reinterpret_cast<const float2 *>(buf + u * PHS + 2 * jrp);
          const float4 wv = *reinterpret_cast<const float4 *>(wb + u * Cip);
          jp[0][0] = fmaf(av.x, wv.x, jp[0][0]); jp[0][1] = fmaf(av.x, wv.y, jp[0][1]); jp[0][2] = fmaf(av.x, wv.z, jp[0][2]); jp[0][3] = fmaf(av.x, wv.w, jp[0][3]);
          jp[1][0] = fmaf(av.y, wv.x, jp[1][0]); jp[1][1] = fmaf(av.y, wv.y, jp[1][1]); jp[1][2] = fmaf(av.y, wv.z, jp[1][2]); jp[1][3] = fmaf(av.y, wv.w, jp[1][3]);
        }
      };
      // 5a. dz1 partial sums: on the stage-to-stage path
      stage_to(buf0, dar);
      __syncthreads();               // every thread is past step 3: buffer 1 (= dlin) is free
      stage_to(buf1, dau);
      acc_j(buf0, 0);
      __syncthreads();
      stage_to(buf0, dan);
      acc_j(buf1, 1);
      __syncthreads();
      acc_j(buf0, 2);
      if (jact) {
        const int dest = (2 * jrp) / PRH, lr = (2 * jrp) % PRH;
        float *ob = (dest == c ? sm : peer) + pl.dz1 + c * PRH * PZ1 + lr * PZ1 + 4 * jcq;
        *reinterpret_cast<float4 *>(ob) = make_float4(jp[0][0], jp[0][1], jp[0][2], jp[0][3]);
        *reinterpret_cast<float4 *>(ob + PZ1) = make_float4(jp[1][0], jp[1][1], jp[1][2], jp[1][3]);
      }
      TSTAMPB(5);
      cluster.sync();  // X2: partial sums exchanged
      TSTAMPB(6);

      // ---- 6. finish d(1x1 conv output), dy = dzf @ W^T, ActNorm backward (modules.py:45-66) ------------------------------
      for (int e = tid; e < PRH * Ci; e += PNT) {
        const int r = e / Ci, i = e - r * Ci;
        dzf[r * pC + i] += dz1[r * PZ1 + i] + dz1[PRH * PZ1 + r * PZ1 + i];
      }
      __syncthreads();
      if (kact) {
        float dy[2][4];
#pragma unroll
        for (int i = 0; i < 2; ++i) dy[i][0] = dy[i][1] = dy[i][2] = dy[i][3] = 0.f;
        const float *x0p = dzf + (2 * krp) * pC, *x1p = x0p + pC;
#pragma unroll 4
        for (int kk = 0; kk < C; ++kk) {
          const float a0 = x0p[kk], a1 = x1p[kk];
          const float4 wv = *reinterpret_cast<const float4 *>(wT + kk * Cp + 4 * kcq);
          dy[0][0] = fmaf(a0, wv.x, dy[0][0]); dy[0][1] = fmaf(a0, wv.y, dy[0][1]); dy[0][2] = fmaf(a0, wv.z, dy[0][2]); dy[0][3] = fmaf(a0, wv.w, dy[0][3]);
          dy[1][0] = fmaf(a1, wv.x, dy[1][0]); dy[1][1] = fmaf(a1, wv.y, dy[1][1]); dy[1][2] = fmaf(a1, wv.z, dy[1][2]); dy[1][3] = fmaf(a1, wv.w, dy[1][3]);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int r = 2 * krp + i;
          if (r < nmy) {
            const size_t off = (cell * B + row0 + lr0 + r) * C + 4 * kcq;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              if (4 * kcq + j < C) {
                const float dxv = dy[i][j] * ans[4 * kcq + j];
                gab[j] += dxv;
                gal[j] += dy[i][j] * yv[i][j];
                if (k > 0) a.dx[off + j] = dxv;
                else if (DXIN) a.dx_in[off + j] = dxv;  // stage 0 (cell == t): gradient of the flow input
              }
            }
          }
        }
      }
      if (k > 0) {
        __syncthreads();
        if (tid == 0) st_release_gpu_b(my_flag, it + 1);  // release at gpu scope, cumulative over the CTA barrier above
      }
      // stash of the weight-gradient operands (dO, dzf: fp32 and planes): off the stage-to-stage path
      for (int e = tid; e < nmy * Co; e += PNT) {
        const int r = e / Co, j = e - r * Co;
        const size_t o = (cell * B + row0 + lr0 + r) * Co + j;
        if (a.dO) a.dO[o] = dor[r * pO + j];
        if (a.pdO_hi) put_plane(a.pdO_hi, a.pdO_lo, o, dor[r * pO + j]);
      }
      for (int e = tid; e < nmy * C; e += PNT) {
        const int r = e / C, j = e - r * C;
        const size_t o = (cell * B + row0 + lr0 + r) * C + j;
        if (a.dzf) a.dzf[o] = dzf[r * pC + j];
        if (a.pdzf_hi) put_plane(a.pdzf_hi, a.pdzf_lo, o, dzf[r * pC + j]);
      }
      TSTAMPB(7);
      // 5b. dh_prev partial sums: needed by this stage's next frame only, so they run after the hand-off to stage k-1.
      //     Buffer 1 still holds dau; buffer 0 (dan) is free since X2.
      stage_to(buf0, dar);
      acc_i(buf1, 1);
      __syncthreads();
      stage_to(buf1, dnr);
      acc_i(buf0, 0);
      __syncthreads();
      acc_i(buf1, 2);
#pragma unroll
      for (int x = 0; x < 2; ++x) {
        float *pq = peer + pl.dhc + (u0 + x) * PHS + 8 * rg;
        *reinterpret_cast<float4 *>(pq) = make_float4(ip[0][2 + x], ip[1][2 + x], ip[2][2 + x], ip[3][2 + x]);
        *reinterpret_cast<float4 *>(pq + 4) = make_float4(ip[4][2 + x], ip[5][2 + x], ip[6][2 + x], ip[7][2 + x]);
#pragma unroll
        for (int r = 0; r < 8; ++r) carry[r][x] += ip[r][x];
      }
      // X3 (split): this CTA is done with both staging buffers and has delivered the peer's dh_prev share
      asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
      x3_pending = true;
      TSTAMPB(8);
    }
    if (x3_pending) { asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory"); x3_pending = false; }
  }

  if (timing)
    printf("core_bwd_pipe stage %d: frames %d cycles/frame: stash prefetch+wait %lld | coupling bwd+dlin %lld | X1 %lld | dh=dlin Wf %lld | gate bwd+dG/dAh stores %lld | dz1 products %lld | X2 %lld | dzf, 1x1 bwd, publish %lld | dh_prev products %lld\n",
           k, it, tacc[0] / it, tacc[1] / it, tacc[2] / it, tacc[3] / it, tacc[4] / it, tacc[5] / it, tacc[6] / it, tacc[7] / it, tacc[8] / it);
  // ---- flush the per-channel gradients -------------------------------------------------------------------------------
#pragma unroll
  for (int g = 0; g < 3; ++g)
#pragma unroll
    for (int x = 0; x < 2; ++x) {
      atomicAdd(&a.g_b_hh[(size_t)k * GH + g * H + uo + x], gbhh[g][x]);
      if (a.g_b_ih) atomicAdd(&a.g_b_ih[(size_t)k * GH + g * H + uo + x], g == 2 ? gbin[x] : gbhh[g][x]);
    }
  if (lane < Cz) {
    if (d.affine) {
      atomicAdd(&a.g_bf[(size_t)k * Co + 2 * lane], gbf[0] * e3[2 * lane]);
      atomicAdd(&a.g_bf[(size_t)k * Co + 2 * lane + 1], gbf[1] * e3[2 * lane + 1]);
      atomicAdd(&a.g_lf[(size_t)k * Co + 2 * lane], 3.0f * glf[0]);
      atomicAdd(&a.g_lf[(size_t)k * Co + 2 * lane + 1], 3.0f * glf[1]);
    } else {
      atomicAdd(&a.g_bf[(size_t)k * Co + lane], gbf[0] * e3[lane]);
      atomicAdd(&a.g_lf[(size_t)k * Co + lane], 3.0f * glf[0]);
    }
  }
  if (kact) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (4 * kcq + j < C) {
        atomicAdd(&a.g_an_bias[(size_t)k * C + 4 * kcq + j], gab[j]);
        atomicAdd(&a.g_an_logs[(size_t)k * C + 4 * kcq + j], gal[j]);
      }
  }
}

// ------------------------------------------------------------------------------------------------
int pipe_bwd_smem_bytes(const Dims &d) { return plan_pipe_bwd(d).total * (int)sizeof(float); }

int launch_bwd_pipe(const BwdArgs &a, cudaStream_t st) {
  static const int timing = getenv("LFI_CORE_TIMING") ? atoi(getenv("LFI_CORE_TIMING")) : 0;
  if (timing) cudaMemcpyToSymbolAsync(g_core_timing_b, &timing, sizeof(int), 0, cudaMemcpyHostToDevice, st);
  auto kern = a.dx_in ? core_bwd_pipe<true> : core_bwd_pipe<false>;
  return launch_pipe(kern, a, PNT, pipe_bwd_smem_bytes(a.d), a.d.K, a.d.K + 1, "core_bwd_pipe", st);
}

}  // namespace core
}  // namespace lfi
