// Persistent stage-pipelined flow core, forward direction (see core_pipe.cuh for the scheme).
#include "core_pipe.cuh"
#include <cooperative_groups.h>
#include <cstdlib>

namespace cg = cooperative_groups;

namespace lfi {
namespace core {

__device__ __forceinline__ int ld_acquire_gpu(const int *p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(int *p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}

// grid = (2, number of steps, pipelines); cluster = the two CTAs along x.
// kCarry: every tile starts from the state a.h0 [K][B][H] and leaves its last frame's state in a.h_last [K][B][H] (time-chunked
// evaluation, lfi_seq_eval); there is no st_h stash.  The instantiation without it starts from zeros and stores st_h.
template <bool kCarry>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(PNT, 1)
core_fwd_pipe(const FwdArgs a, const int P, const int ntiles, int *progress) {
  extern __shared__ __align__(16) float sm[];
  cg::cluster_group cluster = cg::this_cluster();
  const Dims &d = a.d;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = (int)cluster.block_rank();
  const int stage = blockIdx.y, nk = gridDim.y, k = a.k_first + stage, p = blockIdx.z;
  const int C = d.C, Ci = d.Ci, Cz = d.Cz, Co = d.Co, H = d.H, GH = d.GH, B = a.B, Tp = a.Tp, Cp = d.Cp, Cop = d.Cop;
  const PipePlan pl = plan_pipe(d);
  const int pC = pl.pC, pO = pl.pO;
  float *whh = sm + pl.whh, *wz = sm + pl.wz, *wf = sm + pl.wf, *wsm = sm + pl.w;
  float *anb = sm + pl.vec, *ans = anb + C, *bhh = ans + C, *bfs = bhh + 3 * PUC, *e3 = bfs + Co;
  float *hs = sm + pl.h, *z1 = sm + pl.z1, *xs = sm + pl.xs, *zrow = sm + pl.zrow, *osm = sm + pl.o;
  float *peer = cluster.map_shared_rank(sm, c ^ 1);
  const StepWeights w = a.dv.step(d, k);
  const bool first = (k == a.k_first), last = (k == a.k_last);

  // ---- resident weights -------------------------------------------------------------------------
  for (int e = tid; e < H * 3 * (PUC / 4); e += PNT) {
    const int i = e / (3 * (PUC / 4)), rem = e - i * (3 * (PUC / 4)), g = rem / (PUC / 4), u4 = rem - g * (PUC / 4);
    *reinterpret_cast<float4 *>(whh + (i * 3 + g) * PUC + 4 * u4) =
        *reinterpret_cast<const float4 *>(w.WhhT + (size_t)i * GH + g * H + PUC * c + 4 * u4);
  }
  for (int e = tid; e < Ci * 3 * (PUC / 4); e += PNT) {
    const int i = e / (3 * (PUC / 4)), rem = e - i * (3 * (PUC / 4)), g = rem / (PUC / 4), u4 = rem - g * (PUC / 4);
    *reinterpret_cast<float4 *>(wz + (i * 3 + g) * PUC + 4 * u4) =
        *reinterpret_cast<const float4 *>(w.WzT + (size_t)i * GH + g * H + PUC * c + 4 * u4);
  }
  for (int e = tid; e < PUC * (Cop / 4); e += PNT)
    *reinterpret_cast<float4 *>(wf + 4 * e) = *reinterpret_cast<const float4 *>(w.WfT + (size_t)PUC * c * Cop + 4 * e);
  for (int e = tid; e < C * (Cp / 4); e += PNT)
    *reinterpret_cast<float4 *>(wsm + 4 * e) = *reinterpret_cast<const float4 *>(w.Wfwd + 4 * e);
  for (int e = tid; e < C; e += PNT) { anb[e] = w.an_bias[e]; ans[e] = expf(w.an_logs[e]); }
  for (int e = tid; e < 3 * PUC; e += PNT) bhh[e] = w.b_hh[(e / PUC) * H + PUC * c + (e % PUC)];
  for (int e = tid; e < Co; e += PNT) { bfs[e] = w.bf[e]; e3[e] = expf(3.0f * w.lf[e]); }
  cluster.sync();  // both CTAs of the cluster are running before the first distributed-shared-memory access

  // gate tiles: thread owns rows 8rg..8rg+7 x local hidden units u0, u0+1 (all three gates)
  const int ul = (warp & 3) * 8 + (lane & 7), rg = (warp >> 2) * 4 + (lane >> 3);
  const int u0 = 2 * ul;
  const int lr0 = PRH * c;  // first tile row of this CTA's row half
  const int *wait_flag = progress + ((size_t)(p * nk + stage - 1) * 2 + c);
  int *my_flag = progress + ((size_t)(p * nk + stage) * 2 + c);
  int it = 0;

  for (int tile = p; tile < ntiles; tile += P) {
    const int row0 = tile * PR, nrows = min(PR, B - row0);
    const int nmy = max(0, min(PRH, nrows - lr0));
    float hreg[8][2];
    if constexpr (kCarry) {
      // the carried state of this thread's rows and units, into both CTAs' h (the per-frame update's layout); rows past the
      // batch are zero.  The two CTAs together write every unit and row of h, so nothing is zeroed first.
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const bool ok = 8 * rg + r < nrows;
        const float *src = a.h0 + ((size_t)k * B + row0 + 8 * rg + r) * H + PUC * c + u0;
        const float2 v = ok ? *reinterpret_cast<const float2 *>(src) : make_float2(0.f, 0.f);
        hreg[r][0] = v.x; hreg[r][1] = v.y;
      }
#pragma unroll
      for (int x = 0; x < 2; ++x) {
        const float4 v0 = make_float4(hreg[0][x], hreg[1][x], hreg[2][x], hreg[3][x]);
        const float4 v1 = make_float4(hreg[4][x], hreg[5][x], hreg[6][x], hreg[7][x]);
        const int off = pl.h + (PUC * c + u0 + x) * PHS + 8 * rg;
        *reinterpret_cast<float4 *>(sm + off) = v0;
        *reinterpret_cast<float4 *>(sm + off + 4) = v1;
        *reinterpret_cast<float4 *>(peer + off) = v0;
        *reinterpret_cast<float4 *>(peer + off + 4) = v1;
      }
      cluster.sync();  // both halves of the state are in both CTAs before the first recurrent product
    } else {
#pragma unroll
      for (int r = 0; r < 8; ++r) hreg[r][0] = hreg[r][1] = 0.f;
      for (int e = tid; e < H * PHS; e += PNT) hs[e] = 0.f;  // models.py:196-202: state None = zeros
      __syncthreads();
    }

    for (int t = 0; t < Tp; ++t, ++it) {
      const size_t cell = (size_t)k * Tp + t;
      // ---- 0. If stage k-1 has already published this frame (the common case: it runs ahead), request the input now so
      //         that its latency hides behind the recurrent product; otherwise it is fetched after the wait below.
      constexpr int XI = (PRH * 64 + PNT - 1) / PNT;  // C <= 64
      float xv[XI];
      bool have_x = first || ld_acquire_gpu(wait_flag) > it;
      have_x = __syncthreads_and(have_x);   // uniform decision (also orders the previous frame's shared-memory traffic)
      auto fetch_x = [&]() {
#pragma unroll
        for (int i = 0; i < XI; ++i) {
          const int e = tid + PNT * i, r = e / C, cc = e - r * C;
          xv[i] = 0.f;
          if (e < PRH * C && r < nmy) {
            const int b = row0 + lr0 + r;
            xv[i] = first ? a.x0[(size_t)b * a.x_sb + (size_t)t * a.x_st + cc] : __ldcg(a.xin + (cell * B + b) * C + cc);
          }
        }
      };
      if (have_x) fetch_x();
      //         prefetch the gate-ih pre-activations; recurrent product h . W_hh^T (no dependence on stage k-1)
      float2 gp[8][3];
      {
        const float *Gb = a.G + ((size_t)t * B + row0 + 8 * rg) * a.g_ld + (size_t)(k - a.g_k0) * GH + PUC * c + u0;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          if (8 * rg + r < nrows) {
#pragma unroll
            for (int g = 0; g < 3; ++g) gp[r][g] = __ldg(reinterpret_cast<const float2 *>(Gb + (size_t)r * a.g_ld + g * H));
          } else {
#pragma unroll
            for (int g = 0; g < 3; ++g) gp[r][g] = make_float2(0.f, 0.f);
          }
        }
      }
      float ar[8][2], au[8][2], anh[8][2];
      {
        const float2 b0 = *reinterpret_cast<const float2 *>(bhh + u0), b1 = *reinterpret_cast<const float2 *>(bhh + PUC + u0),
                     b2 = *reinterpret_cast<const float2 *>(bhh + 2 * PUC + u0);
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          ar[r][0] = b0.x; ar[r][1] = b0.y; au[r][0] = b1.x; au[r][1] = b1.y; anh[r][0] = b2.x; anh[r][1] = b2.y;
        }
      }
#pragma unroll 4
      for (int kk = 0; kk < H; ++kk) {
        const float4 a0 = *reinterpret_cast<const float4 *>(hs + kk * PHS + 8 * rg);
        const float4 a1 = *reinterpret_cast<const float4 *>(hs + kk * PHS + 8 * rg + 4);
        const float2 wr = *reinterpret_cast<const float2 *>(whh + (kk * 3 + 0) * PUC + u0);
        const float2 wu = *reinterpret_cast<const float2 *>(whh + (kk * 3 + 1) * PUC + u0);
        const float2 wn = *reinterpret_cast<const float2 *>(whh + (kk * 3 + 2) * PUC + u0);
        const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          ar[r][0] = fmaf(av[r], wr.x, ar[r][0]); ar[r][1] = fmaf(av[r], wr.y, ar[r][1]);
          au[r][0] = fmaf(av[r], wu.x, au[r][0]); au[r][1] = fmaf(av[r], wu.y, au[r][1]);
          anh[r][0] = fmaf(av[r], wn.x, anh[r][0]); anh[r][1] = fmaf(av[r], wn.y, anh[r][1]);
        }
      }

      // ---- 1. wait for stage k-1, ActNorm (modules.py:45-66) on this CTA's 32 rows ---------------------------------
      if (!have_x) {
        if (tid == 0) {
          spin_wait_gt(wait_flag, it);
        }
        __syncthreads();
        fetch_x();
      }
#pragma unroll
      for (int i = 0; i < XI; ++i) {
        const int e = tid + PNT * i, r = e / C, cc = e - r * C;
        if (e < PRH * C) {
          float v = 0.f;
          if (r < nmy) {
            const int b = row0 + lr0 + r;
            v = (xv[i] + anb[cc]) * ans[cc];
            if (a.st_y) a.st_y[(cell * B + b) * C + cc] = v;
            if (a.py_hi) put_plane(a.py_hi, a.py_lo, (cell * B + b) * C + cc, v);
          }
          xs[r * pC + cc] = v;
        }
      }
      __syncthreads();
      // ---- 2. invertible 1x1 conv (modules.py:186): z = y @ W, 2 rows x 4 columns per thread -------------------------
      {
        const int ncq = Cp >> 2;
        if (tid < 16 * ncq) {
          const int cq = tid % ncq, rp = tid / ncq;
          float z[2][4];
#pragma unroll
          for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) z[i][j] = 0.f;
          const float *x0p = xs + (2 * rp) * pC, *x1p = x0p + pC;
#pragma unroll 4
          for (int kk = 0; kk < C; ++kk) {
            const float a0 = x0p[kk], a1 = x1p[kk];
            const float4 wv = *reinterpret_cast<const float4 *>(wsm + kk * Cp + 4 * cq);
            z[0][0] = fmaf(a0, wv.x, z[0][0]); z[0][1] = fmaf(a0, wv.y, z[0][1]); z[0][2] = fmaf(a0, wv.z, z[0][2]); z[0][3] = fmaf(a0, wv.w, z[0][3]);
            z[1][0] = fmaf(a1, wv.x, z[1][0]); z[1][1] = fmaf(a1, wv.y, z[1][1]); z[1][2] = fmaf(a1, wv.z, z[1][2]); z[1][3] = fmaf(a1, wv.w, z[1][3]);
          }
#pragma unroll
          for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (4 * cq + j < C) zrow[(2 * rp + i) * pC + 4 * cq + j] = z[i][j];
        }
      }
      __syncthreads();
      for (int e = tid; e < Ci * PRH; e += PNT) {  // z1 in act layout, to both CTAs of the cluster
        const int j = e / PRH, r = e - j * PRH;
        const float v = zrow[r * pC + j];
        z1[j * PHS + lr0 + r] = v;
        peer[pl.z1 + j * PHS + lr0 + r] = v;
      }
      if (a.st_zf)
        for (int e = tid; e < nmy * C; e += PNT) {
          const int r = e / C, j = e - r * C;
          const size_t o = (cell * B + row0 + lr0 + r) * C + j;
          a.st_zf[o] = zrow[r * pC + j];
          if (a.pzf_hi) put_plane(a.pzf_hi, a.pzf_lo, o, zrow[r * pC + j]);
        }
      cluster.sync();  // A: z1 complete in both CTAs; both are done reading h of the previous frame

      // ---- 3. z1 part of the gate-ih product, GRU gate math (torch nn.GRUCell, gate order r, z, n) ------------------
      float ani[8][2];
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        ar[r][0] += gp[r][0].x; ar[r][1] += gp[r][0].y; au[r][0] += gp[r][1].x; au[r][1] += gp[r][1].y;
        ani[r][0] = gp[r][2].x; ani[r][1] = gp[r][2].y;
      }
#pragma unroll 4
      for (int kk = 0; kk < Ci; ++kk) {
        const float4 a0 = *reinterpret_cast<const float4 *>(z1 + kk * PHS + 8 * rg);
        const float4 a1 = *reinterpret_cast<const float4 *>(z1 + kk * PHS + 8 * rg + 4);
        const float2 wr = *reinterpret_cast<const float2 *>(wz + (kk * 3 + 0) * PUC + u0);
        const float2 wu = *reinterpret_cast<const float2 *>(wz + (kk * 3 + 1) * PUC + u0);
        const float2 wn = *reinterpret_cast<const float2 *>(wz + (kk * 3 + 2) * PUC + u0);
        const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          ar[r][0] = fmaf(av[r], wr.x, ar[r][0]); ar[r][1] = fmaf(av[r], wr.y, ar[r][1]);
          au[r][0] = fmaf(av[r], wu.x, au[r][0]); au[r][1] = fmaf(av[r], wu.y, au[r][1]);
          ani[r][0] = fmaf(av[r], wn.x, ani[r][0]); ani[r][1] = fmaf(av[r], wn.y, ani[r][1]);
        }
      }
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int x = 0; x < 2; ++x) {
          const float rgt = fast_sigmoid(ar[r][x]), ugt = fast_sigmoid(au[r][x]);
          const float ng = fast_tanh(ani[r][x] + rgt * anh[r][x]);
          ar[r][x] = rgt; au[r][x] = ugt; ani[r][x] = ng;
          hreg[r][x] = ng + ugt * (hreg[r][x] - ng);
        }
      {  // stash for the backward pass (gates post-activation, h-side n pre-activation, new state)
        const size_t rb = cell * B + row0 + 8 * rg;
        const int uo = PUC * c + u0;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          if (8 * rg + r < nrows) {
            if (a.st_gates) {
              float *gq = a.st_gates + (rb + r) * GH + uo;
              *reinterpret_cast<float2 *>(gq) = make_float2(ar[r][0], ar[r][1]);
              *reinterpret_cast<float2 *>(gq + H) = make_float2(au[r][0], au[r][1]);
              *reinterpret_cast<float2 *>(gq + 2 * H) = make_float2(ani[r][0], ani[r][1]);
            }
            if (a.st_ahn) *reinterpret_cast<float2 *>(a.st_ahn + (rb + r) * H + uo) = make_float2(anh[r][0], anh[r][1]);
            if constexpr (kCarry) {
              if (t == Tp - 1)
                *reinterpret_cast<float2 *>(a.h_last + ((size_t)k * B + row0 + 8 * rg + r) * H + uo) = make_float2(hreg[r][0], hreg[r][1]);
            } else {
              *reinterpret_cast<float2 *>(a.st_h + (rb + r) * H + uo) = make_float2(hreg[r][0], hreg[r][1]);
            }
            if (a.ph_hi) put_plane2(a.ph_hi, a.ph_lo, (rb + r) * H + uo, hreg[r][0], hreg[r][1]);
          }
        }
      }
#pragma unroll
      for (int x = 0; x < 2; ++x) {  // new state into both CTAs' h (act layout)
        const float4 v0 = make_float4(hreg[0][x], hreg[1][x], hreg[2][x], hreg[3][x]);
        const float4 v1 = make_float4(hreg[4][x], hreg[5][x], hreg[6][x], hreg[7][x]);
        const int off = pl.h + (PUC * c + u0 + x) * PHS + 8 * rg;
        *reinterpret_cast<float4 *>(sm + off) = v0;
        *reinterpret_cast<float4 *>(sm + off + 4) = v1;
        *reinterpret_cast<float4 *>(peer + off) = v0;
        *reinterpret_cast<float4 *>(peer + off + 4) = v1;
      }
      __syncthreads();

      // ---- 4. LinearZeros (modules.py:93-95), partial sum over this CTA's 64 hidden units, all 64 rows ---------------
      {
        const int ncoq = Cop >> 2;
        if (tid < 16 * ncoq) {
          const int cq = tid % ncoq, rq = tid / ncoq;
          float o[4][4];
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) o[i][j] = 0.f;
          const float *hb = hs + (PUC * c) * PHS + 4 * rq;
#pragma unroll 4
          for (int u = 0; u < PUC; ++u) {
            const float4 av = *reinterpret_cast<const float4 *>(hb + u * PHS);
            const float4 wv = *reinterpret_cast<const float4 *>(wf + u * Cop + 4 * cq);
            const float a4[4] = {av.x, av.y, av.z, av.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              o[i][0] = fmaf(a4[i], wv.x, o[i][0]); o[i][1] = fmaf(a4[i], wv.y, o[i][1]);
              o[i][2] = fmaf(a4[i], wv.z, o[i][2]); o[i][3] = fmaf(a4[i], wv.w, o[i][3]);
            }
          }
          const int dest = (4 * rq) / PRH, lr = (4 * rq) % PRH;  // CTA that owns these rows; slot c holds this CTA's partial
          float *ob = (dest == c ? sm : peer) + pl.o + c * PRH * pO + lr * pO + 4 * cq;
#pragma unroll
          for (int i = 0; i < 4; ++i) *reinterpret_cast<float4 *>(ob + i * pO) = make_float4(o[i][0], o[i][1], o[i][2], o[i][3]);
        }
      }
      cluster.sync();  // B: partial sums and the new state are complete in both CTAs

      // ---- 5. affine coupling (models.py:331-341), log-det, NLL on the last step (modules.py:207-212, models.py:563-565)
      {
        const float *o0 = osm, *o1 = osm + PRH * pO;
        float ldv = 0.f;  // running log-det of row warp + 8 * lane: one round trip for the warp's rows
        if ((!first || a.ld_accumulate) && warp + (PNT / 32) * lane < nmy)
          ldv = __ldcg(a.ld + (size_t)t * B + row0 + lr0 + warp + (PNT / 32) * lane);
        for (int r = warp, n = 0; r < nmy; r += PNT / 32, ++n) {
          const int b = row0 + lr0 + r;
          float lsum = 0.f;
          for (int q = lane; q < Cz; q += 32) {
            const float z2 = zrow[r * pC + Ci + q];
            if (d.affine) {
              const float shift = (o0[r * pO + 2 * q] + o1[r * pO + 2 * q] + bfs[2 * q]) * e3[2 * q];
              const float sc = (o0[r * pO + 2 * q + 1] + o1[r * pO + 2 * q + 1] + bfs[2 * q + 1]) * e3[2 * q + 1];
              const float s = fmaxf(sigmoidf_(sc + 2.0f), d.eps);
              zrow[r * pC + Ci + q] = (z2 + shift) * s;
              lsum += logf(s);
              if (a.st_o) *reinterpret_cast<float2 *>(a.st_o + (cell * B + b) * Co + 2 * q) = make_float2(shift, sc);
              if (a.scale_out && t == Tp - 1) a.scale_out[((size_t)k * B + b) * Cz + q] = s;
            } else {
              const float ov = (o0[r * pO + q] + o1[r * pO + q] + bfs[q]) * e3[q];
              zrow[r * pC + Ci + q] = z2 + ov;
              if (a.st_o) a.st_o[(cell * B + b) * Co + q] = ov;
            }
          }
          lsum = warp_sum(lsum);
          __syncwarp();
          const float ld = lsum + __shfl_sync(0xffffffffu, ldv, n);
          if (last && a.nll) {
            float zsq = 0.f;
            for (int cc = lane; cc < C; cc += 32) { const float z = zrow[r * pC + cc]; zsq += z * z; }
            zsq = warp_sum(zsq);
            if (lane == 0) a.nll[(size_t)t * B + b] = -(ld - 0.5f * (zsq + (float)C * kLog2Pi)) / kLn2;
          }
          if (lane == 0) a.ld[(size_t)t * B + b] = ld;
        }
      }
      __syncthreads();
      {
        float *dst = last ? a.z_out + (size_t)t * B * C : a.xin + (cell + Tp) * B * C;  // XIN[k+1][t]
        for (int e = tid; e < nmy * C; e += PNT) { const int r = e / C, j = e - r * C; dst[(size_t)(row0 + lr0 + r) * C + j] = zrow[r * pC + j]; }
      }
      if (!last) {
        __syncthreads();
        if (tid == 0) { __threadfence(); st_release_gpu(my_flag, it + 1); }
      }
    }
    cluster.sync();  // the peer may still be reading this CTA's partial sums / writing state of the tile's last frame
  }
}

// ------------------------------------------------------------------------------------------------
constexpr int kPipeMaxSmem = 227 * 1024;

bool pipe_supported(const Dims &d, bool bwd) {
  if (d.G != 3 || d.H != 2 * PUC) return false;
  if (d.C > 64 || d.Co > 64 || d.C < 2) return false;
  if (d.affine && (d.Co & 1)) return false;
  if (2 * d.K > sm_count()) return false;
  if (d.Ci > 32 || d.Cz > 32) return false;
  const int bytes = bwd ? pipe_bwd_smem_bytes(d) : plan_pipe(d).total * (int)sizeof(float);
  return bytes <= kPipeMaxSmem;
}

int launch_fwd_pipe(const FwdArgs &a, cudaStream_t st) {
  const int nk = a.k_last - a.k_first + 1;
  const int smem = plan_pipe(a.d).total * (int)sizeof(float);
  if (a.h0 || a.h_last) {
    LFI_REQUIRE(a.h0 && a.h_last, LFI_ERR_ARG, "core_fwd_pipe: a carried state needs both h0 and h_last");
    return launch_pipe(core_fwd_pipe<true>, a, PNT, smem, nk, nk, "core_fwd_pipe", st);
  }
  return launch_pipe(core_fwd_pipe<false>, a, PNT, smem, nk, nk, "core_fwd_pipe", st);
}

}  // namespace core
}  // namespace lfi
