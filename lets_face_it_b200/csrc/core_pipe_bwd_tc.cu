// Persistent stage-pipelined flow core, backward direction, gate-gradient products on the tensor cores (tensor-core GEMM
// modes).  Same pipeline as core_pipe_bwd.cu (stage k = one 2-CTA cluster walking the frames in reverse, cell (k, t)
// consumes d(output of step k) published by stage k+1, carries d h[k][t] across frames, publishes d(input) to stage
// k-1; each CTA owns 64 hidden units = 192 gate columns), with its three large products as tcgen05.mma on split-bf16
// operands (three products, fp32-grade; fp32 accumulation in TMEM):
//   P1  dh      += dlin  Wf[:, own units]          [64 x 56]  x [56 x 64]    LinearZeros backward (modules.py:93-95)
//   P2  dz1      = dA_i  W_ih[own gates, :Ci]      [64 x 192] x [192 x 28]   partial over this CTA's gate columns
//   P3  dh_prev  = dA_h  W_hh[own gates, :]        [64 x 192] x [192 x 128]  partial; own units stay, the rest goes to the peer
// The weight slices are resident as (hi, lo) planes in the swizzled K-major UMMA layout; dlin and the gate gradients
// dA = (d a_r, d a_u, d a_n | r d a_n) are written as planes by the threads that produce them.  Thread = one sequence x 16
// hidden units (TMEM lane = sequence; every product is issued a second time with the A descriptor moved back by 64 rows so
// that lanes 64..127 carry the other half of the columns), which also makes the reads of the tiled gate stash contiguous.
// A ninth warp issues every MMA, so the issue latency of ~130 instructions per frame stays off the stage-to-stage path.
// Reference: autograd of FlowStep.normal_flow (models.py:311-342) and of nn.GRUCell inside f_seq.forward (models.py:204-214).
#include "core_pipe.cuh"
#include "tc_ptx.cuh"
#include <cooperative_groups.h>
#include <cstdlib>

namespace cg = cooperative_groups;

namespace lfi {
namespace core {

using namespace tcp;

namespace {

__device__ __forceinline__ void st_release_gpu_bt(int *p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void csync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }           // the eight compute warps
__device__ __forceinline__ void bar_arrive(int id) { asm volatile("bar.arrive %0, 288;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void bar_sync_all(int id) { asm volatile("bar.sync %0, 288;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory"); }

constexpr int BNT = 288;  // eight compute warps + the MMA-issue warp
// byte offsets of the operand blocks (1024-byte aligned)
constexpr int kBH = 0;                     // W_hh slice [n = 128 units][k = 192 own gate columns]: 2 planes x 3 k-blocks x [128 x 128 B]
constexpr int kBHPlane = 3 * 128 * 128;
constexpr int kBZ = kBH + 2 * kBHPlane;    // W_ih slice [n = 32 (Ci)][k = 192]:                     2 planes x 3 k-blocks x [32 x 128 B]
constexpr int kBZPlane = 3 * 32 * 128;
constexpr int kBF = kBZ + 2 * kBZPlane;    // Wf slice   [n = 64 own units][k = 64 (Co)]:            2 planes x [64 x 128 B]
constexpr int kBFPlane = 64 * 128;
constexpr int kADA = kBF + 2 * kBFPlane;   // gate gradients [64 rows][k = 3 x 64]: 2 planes x 3 k-blocks x [64 x 128 B]; block 0 doubles as dlin
constexpr int kADAPlane = 3 * 64 * 128;
constexpr int kF32 = kADA + 2 * kADAPlane;
constexpr int kTmemCols = 256;
constexpr int kColLZ = 0, kColHP = 64, kColZ = 192;  // accumulators: dlin Wf (2 x 32), dh_prev (2 x [32 own | 32 peer]), dz1 (32)

struct PlanBT {
  int wT, vec, dzf, dz1x, dhc, bars, total;
  int pC;
};
__host__ __device__ inline PlanBT plan_bt(const Dims &d) {
  PlanBT p;
  p.pC = odd(d.C);
  int o = kF32;
  auto take = [&](int nfloats) { int r = o; o += round_up(nfloats, 4) * 4; return r; };
  p.wT = take(d.C * d.Cp);       // [i][j] = W[j][i]
  p.vec = take(d.C + d.Co);      // exp(an_logs), exp(3 lf)
  p.dzf = take(PRH * p.pC);      // row-major d(1x1 conv output) of this CTA's rows
  p.dz1x = take(PRH * 32);       // the peer's dz1 partial for this CTA's rows
  p.dhc = take(4 * PR * 16);     // the peer's dh_prev partial for this CTA's units: [unit group][row][16]
  p.bars = take(16);
  p.total = o + 1024;
  return p;
}

__device__ int g_core_timing_bt = 0;

}  // namespace

// DXIN: stage 0 also stores the gradient of the flow input (BwdArgs.dx_in); the instantiation without it is the plain backward
template <bool DXIN>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(BNT, 1)
core_bwd_pipe_tc(const BwdArgs a, const int P, const int ntiles, int *progress) {
  extern __shared__ __align__(16) uint8_t smraw[];
  uint8_t *smb = (uint8_t *)(((uintptr_t)smraw + 1023) & ~(uintptr_t)1023);
  cg::cluster_group cluster = cg::this_cluster();
  const Dims &d = a.d;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = (int)cluster.block_rank();
  const int k = blockIdx.y, K = d.K, p = blockIdx.z;
  const int C = d.C, Ci = d.Ci, Cz = d.Cz, Co = d.Co, H = d.H, GH = d.GH, B = a.B, Tp = a.Tp, Cp = d.Cp, Cip = d.Cip;
  const unsigned magC = div_magic(C), magCi = div_magic(Ci);
  const PlanBT pl = plan_bt(d);
  const int pC = pl.pC;
  float *wT = (float *)(smb + pl.wT), *ans = (float *)(smb + pl.vec), *e3 = ans + C;
  float *dzf = (float *)(smb + pl.dzf), *dz1x = (float *)(smb + pl.dz1x), *dhc = (float *)(smb + pl.dhc);
  uint64_t *bar1 = (uint64_t *)(smb + pl.bars), *bar2 = bar1 + 1, *bar3 = bar1 + 2;
  uint32_t *tmem_slot = (uint32_t *)(bar1 + 3);
  uint8_t *peerb = cluster.map_shared_rank(smb, c ^ 1);
  const StepWeights w = a.dv.step(d, k);
  const bool lastk = (k == K - 1);
  const bool mma_warp = warp == 8;

  // ---- resident weights: fp32 -> (hi, lo) bf16 planes in the K-major swizzled UMMA layout ------------------------
  // P3: row n' = hf*64 + pe*32 + i  <->  hidden unit m = 64 (pe ? 1-c : c) + 32 hf + i ;  k = g*64 + u  <->  W_hh[g*H + 64c + u][m]
  for (int e = tid; e < 128 * 24; e += BNT) {
    const int np = e / 24, ch = e - np * 24, g = ch >> 3, u0 = (ch & 7) * 8;
    const int hf = np >> 6, pe = (np >> 5) & 1, i = np & 31;
    const int m = 64 * (pe ? (1 - c) : c) + 32 * hf + i;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = w.Whh[(size_t)(g * H + PUC * c + u0 + j) * H + m];
    uint4 hi, lo;
    split8(v, hi, lo);
    const uint32_t off = (uint32_t)g * (128 * 128) + sw128_off(np, ch & 7);
    *reinterpret_cast<uint4 *>(smb + kBH + off) = hi;
    *reinterpret_cast<uint4 *>(smb + kBH + kBHPlane + off) = lo;
  }
  // P2: row n = z1 column i (zero beyond Ci) ; k = g*64 + u  <->  W_ih[g*H + 64c + u][i]
  for (int e = tid; e < 32 * 24; e += BNT) {
    const int n = e / 24, ch = e - n * 24, g = ch >> 3, u0 = (ch & 7) * 8;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = (n < Ci) ? w.WihZ[(size_t)(g * H + PUC * c + u0 + j) * Cip + n] : 0.f;
    uint4 hi, lo;
    split8(v, hi, lo);
    const uint32_t off = (uint32_t)g * (32 * 128) + sw128_off(n, ch & 7);
    *reinterpret_cast<uint4 *>(smb + kBZ + off) = hi;
    *reinterpret_cast<uint4 *>(smb + kBZ + kBZPlane + off) = lo;
  }
  // P1: row n = own hidden unit u ; k = LinearZeros output j (zero beyond Co)  <->  Wf[j][64c + u]
  for (int e = tid; e < 64 * 8; e += BNT) {
    const int n = e >> 3, ch = e & 7;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = (8 * ch + j < Co) ? w.Wf[(size_t)(8 * ch + j) * H + PUC * c + n] : 0.f;
    uint4 hi, lo;
    split8(v, hi, lo);
    const uint32_t off = sw128_off(n, ch);
    *reinterpret_cast<uint4 *>(smb + kBF + off) = hi;
    *reinterpret_cast<uint4 *>(smb + kBF + kBFPlane + off) = lo;
  }
  for (int e = tid; e < C * (Cp / 4); e += BNT)
    *reinterpret_cast<float4 *>(wT + 4 * e) = *reinterpret_cast<const float4 *>(w.WT + 4 * e);
  for (int e = tid; e < C; e += BNT) ans[e] = expf(w.an_logs[e]);
  for (int e = tid; e < Co; e += BNT) e3[e] = expf(3.0f * w.lf[e]);
  for (int e = tid; e < 2 * kADAPlane / 16; e += BNT) reinterpret_cast<uint4 *>(smb + kADA)[e] = make_uint4(0u, 0u, 0u, 0u);
  if (tid == 0) {
    mbar_init(bar1, 1); mbar_init(bar2, 1); mbar_init(bar3, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (mma_warp) tmem_alloc(tmem_slot, kTmemCols);
  fence_before();
  fence_async_smem();
  cluster.sync();
  fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t sBH = smem_u32(smb + kBH), sBZ = smem_u32(smb + kBZ), sBF = smem_u32(smb + kBF), sADA = smem_u32(smb + kADA);

  // compute threads: TMEM lane L = 32 (warp % 4) + lane <-> sequence L % 64, unit half L / 64; the two warps of a lane quarter
  // split that half's 32 hidden units
  const int q = warp & 3, sub = (warp >> 2) & 1;
  const int L = 32 * q + lane, row = L & 63, half = q >> 1;
  const int ub = 32 * half + 16 * sub, hs = 2 * half + sub;
  const uint32_t tlane = tmem + ((uint32_t)(32 * q) << 16);
  const int lr0 = PRH * c;
  const int ncq = Cp >> 2;
  const int kcq = tid % ncq, krp = tid / ncq;  // 1x1 conv backward: rows 2krp, 2krp+1 x columns 4kcq..
  const bool kact = !mma_warp && krp < PRH / 2;
  const int *wait_flag = progress + ((size_t)(p * K + k + 1) * 2 + c);
  int *my_flag = progress + ((size_t)(p * K + k) * 2 + c);
  int it = 0;
  bool x3_pending = false;
  const bool timing = g_core_timing_bt && tid == 0 && c == 0 && p == 0 && (k == 8 || k == 0 || k == K - 1);
  long long tacc[12] = {0}, tprev = 0;
#define TSTAMPT(i) do { if (timing) { const long long now_ = clock64(); tacc[i] += now_ - tprev; tprev = now_; } } while (0)

  // per-channel gradient accumulators (flushed once at the end); d b_ih / d b_hh are column sums of the dG / dA_h planes this
  // kernel writes and are reduced from them by the caller (aux::colsum_planes, on the weight-gradient stream)
  float gbf[2] = {0.f, 0.f}, glf[2] = {0.f, 0.f};
  float gab[4] = {0.f, 0.f, 0.f, 0.f}, gal[4] = {0.f, 0.f, 0.f, 0.f};

  for (int tile = p; tile < ntiles; tile += P) {
    const int row0 = tile * PR, nrows = min(PR, B - row0);
    const int nmy = max(0, min(PRH, nrows - lr0));
    const bool rowok = row < nrows;
    float carry[16];  // d h[k][t] arriving from frame t+1 (this thread's sequence x 16 units)
#pragma unroll
    for (int j = 0; j < 16; ++j) carry[j] = 0.f;

    for (int t = Tp - 1; t >= 0; --t, ++it) {
      const size_t cell = (size_t)k * Tp + t;
      const uint32_t ph = (uint32_t)(it & 1);

      if (mma_warp) {
        // =================================== MMA-issue warp ===================================
        if (x3_pending) { cluster_wait(); x3_pending = false; }
        cluster_arrive(); cluster_wait();                       // X1: dlin planes of all 64 rows present
        if (lane == 0) {
          fence_after(); fence_async_smem();
          const uint32_t idesc = idesc_bf16_m128(32);
          uint32_t acc = 0;
#pragma unroll
          for (int pr = 0; pr < 3; ++pr) {  // (hi,hi), (hi,lo), (lo,hi)
            const uint32_t pa = (pr == 2) ? kADAPlane : 0, pb = (pr == 1) ? kBFPlane : 0;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
              for (int hf = 0; hf < 2; ++hf)
                umma_bf16(tmem + kColLZ + hf * 32, make_sdesc(sADA + pa + ks * 32 - hf * (64 * 128), 1024, kSw128),
                          make_sdesc(sBF + pb + hf * (32 * 128) + ks * 32, 1024, kSw128), idesc, acc);
              acc = 1;
            }
          }
          umma_commit(bar1);
        }
        __syncwarp();
        bar_sync_all(2);                                        // gate gradients (r, u, n blocks) written
        if (lane == 0) {
          fence_after(); fence_async_smem();
          const uint32_t idesc = idesc_bf16_m128(32);
          uint32_t acc = 0;
#pragma unroll
          for (int pr = 0; pr < 3; ++pr) {
            const uint32_t pa = (pr == 2) ? kADAPlane : 0, pb = (pr == 1) ? kBZPlane : 0;
#pragma unroll
            for (int kb = 0; kb < 3; ++kb)
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                umma_bf16(tmem + kColZ, make_sdesc(sADA + pa + kb * (64 * 128) + ks * 32, 1024, kSw128),
                          make_sdesc(sBZ + pb + kb * (32 * 128) + ks * 32, 1024, kSw128), idesc, acc);
                acc = 1;
              }
          }
          umma_commit(bar2);
        }
        __syncwarp();
        bar_sync_all(3);                                        // n block overwritten with r * d a_n
        cluster_arrive();                                       // X2 (this warp has nothing to publish)
        if (lane == 0) {
          fence_after(); fence_async_smem();
          const uint32_t idesc = idesc_bf16_m128(64);
          uint32_t acc = 0;
#pragma unroll
          for (int pr = 0; pr < 3; ++pr) {
            const uint32_t pa = (pr == 2) ? kADAPlane : 0, pb = (pr == 1) ? kBHPlane : 0;
#pragma unroll
            for (int kb = 0; kb < 3; ++kb)
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
                for (int hf = 0; hf < 2; ++hf)
                  umma_bf16(tmem + kColHP + hf * 64, make_sdesc(sADA + pa + kb * (64 * 128) + ks * 32 - hf * (64 * 128), 1024, kSw128),
                            make_sdesc(sBH + pb + kb * (128 * 128) + hf * (64 * 128) + ks * 32, 1024, kSw128), idesc, acc);
                acc = 1;
              }
          }
          umma_commit(bar3);
        }
        __syncwarp();
        cluster_wait();                                         // X2
        cluster_arrive();                                       // X3 (split)
        x3_pending = true;
        continue;
      }

      // ===================================== compute warps =====================================
      if (timing) tprev = clock64();
      // ---- 0. prefetch the coupling stash of this CTA's rows (the gate stash is requested after X1: its latency hides behind
      //         the LinearZeros-backward product, and the registers stay free until then) ---------------------------------------
      constexpr int NR = PRH / 8;
      float c_dnl[NR], c_z2[NR];
      float2 c_o[NR];
#pragma unroll
      for (int n = 0; n < NR; ++n) {
        const int r = warp + 8 * n, qq = lane;
        c_dnl[n] = 0.f; c_z2[n] = 0.f; c_o[n] = make_float2(0.f, 0.f);
        if (r < nmy) {
          const int b = row0 + lr0 + r;
          c_dnl[n] = a.dnll[(size_t)t * B + b];
          if (qq < Cz) {
            if (d.affine) {
              c_o[n] = *reinterpret_cast<const float2 *>(a.st.o + (cell * B + b) * Co + 2 * qq);
              c_z2[n] = a.st.zf[(cell * B + b) * C + Ci + qq];
            } else {
              c_o[n].x = a.st.o[(cell * B + b) * Co + qq];
            }
          }
        }
      }
      // ---- 1. wait for stage k+1 ---------------------------------------------------------------------------------------
      if (!lastk) {
        if (tid == 0) {
          spin_wait_gt(wait_flag, it);
        }
        csync();
      }
      TSTAMPT(0);
      // ---- 2. coupling backward (models.py:331-341) on this CTA's 32 rows; dlin leaves as operand planes -------------------
      float c_dz[NR], c_dx1[NR];
#pragma unroll
      for (int n = 0; n < NR; ++n) {
        const int r = warp + 8 * n, qq = lane;
        c_dz[n] = 0.f; c_dx1[n] = 0.f;
        if (r < nmy) {
          const int b = row0 + lr0 + r;
          const float *dxp = a.dx + ((cell + Tp) * B + b) * C;
          const float *zp = a.z + ((size_t)t * B + b) * C;
          if (qq < Cz) c_dz[n] = lastk ? c_dnl[n] * zp[Ci + qq] / kLn2 : __ldcg(dxp + Ci + qq);  // last step: d nll / d z = z / ln2
          if (qq < Ci) c_dx1[n] = lastk ? c_dnl[n] * zp[qq] / kLn2 : __ldcg(dxp + qq);
        }
      }
      if (x3_pending) { cluster_wait(); x3_pending = false; }  // the peer is done with the gate-gradient blocks (block 0 = dlin)
#pragma unroll
      for (int n = 0; n < NR; ++n) {
        const int r = warp + 8 * n, qq = lane;
        float dz2 = 0.f, dl0 = 0.f, dl1 = 0.f;
        if (r < nmy && qq < Cz) {
          const float dld = -c_dnl[n] / kLn2;  // d nll / d logdet
          const float dz2n = c_dz[n];
          if (d.affine) {
            const float shift = c_o[n].x, sc = c_o[n].y, z2 = c_z2[n];
            const float sg = fast_sigmoid(sc + 2.0f), s = fmaxf(sg, d.eps);
            const float ds = dz2n * (z2 + shift) + dld / s;
            dz2 = dz2n * s;
            const float dsc = (sg >= d.eps) ? ds * sg * (1.0f - sg) : 0.f;
            gbf[0] += dz2; gbf[1] += dsc; glf[0] += dz2 * shift; glf[1] += dsc * sc;
            dl0 = dz2 * e3[2 * qq]; dl1 = dsc * e3[2 * qq + 1];
          } else {
            const float ov = c_o[n].x;
            dz2 = dz2n;
            gbf[0] += dz2n; glf[0] += dz2n * ov;
            dl0 = dz2n * e3[qq];
          }
        }
        if (qq < Cz) dzf[r * pC + Ci + qq] = dz2;
        if (qq < Ci) dzf[r * pC + qq] = c_dx1[n];
        // dlin of tile row lr0 + r as (hi, lo) planes in both CTAs (rows beyond the batch: zeros), and the dW_f operand stash
        if (d.affine) {
          if (qq < Cz) {
            const __nv_bfloat162 hh = __floats2bfloat162_rn(dl0, dl1);
            const __nv_bfloat162 ll = __floats2bfloat162_rn(dl0 - __low2float(hh), dl1 - __high2float(hh));
            const uint32_t off = kADA + sw128_off(lr0 + r, (2 * qq) >> 3) + ((2 * qq) & 7) * 2;
            *reinterpret_cast<__nv_bfloat162 *>(smb + off) = hh; *reinterpret_cast<__nv_bfloat162 *>(smb + off + kADAPlane) = ll;
            *reinterpret_cast<__nv_bfloat162 *>(peerb + off) = hh; *reinterpret_cast<__nv_bfloat162 *>(peerb + off + kADAPlane) = ll;
            if (r < nmy) {
              const size_t o = (cell * B + row0 + lr0 + r) * Co + 2 * qq;
              if (a.dO) *reinterpret_cast<float2 *>(a.dO + o) = make_float2(dl0, dl1);
              if (a.pdO_hi) {
                *reinterpret_cast<__nv_bfloat162 *>((__nv_bfloat16 *)a.pdO_hi + o) = hh;
                if (a.pdO_lo) *reinterpret_cast<__nv_bfloat162 *>((__nv_bfloat16 *)a.pdO_lo + o) = ll;
              }
            }
          }
        } else if (qq < Cz) {
          const __nv_bfloat16 hh = __float2bfloat16_rn(dl0), ll = __float2bfloat16_rn(dl0 - __bfloat162float(hh));
          const uint32_t off = kADA + sw128_off(lr0 + r, qq >> 3) + (qq & 7) * 2;
          *reinterpret_cast<__nv_bfloat16 *>(smb + off) = hh; *reinterpret_cast<__nv_bfloat16 *>(smb + off + kADAPlane) = ll;
          *reinterpret_cast<__nv_bfloat16 *>(peerb + off) = hh; *reinterpret_cast<__nv_bfloat16 *>(peerb + off + kADAPlane) = ll;
          if (r < nmy) {
            const size_t o = (cell * B + row0 + lr0 + r) * Co + qq;
            if (a.dO) a.dO[o] = dl0;
            if (a.pdO_hi) put_plane(a.pdO_hi, a.pdO_lo, o, dl0);
          }
        }
      }
      fence_async_smem();
      TSTAMPT(1);
      cluster_arrive(); cluster_wait();  // X1: dlin of all 64 rows present in both CTAs (the MMA warp issues P1 now)
      TSTAMPT(2);
      // gate stash of this thread's sequence x 16 units (tiled layout: contiguous over the warp's sequences)
      float4 sr[4], su[4], sn[4], sa[4], sh[4];
      {
        const float *gq = a.st.gates + stash_tiled_off(cell, ntiles, tile, c, hs, 3, 0, 0) + 4 * row;
        const float *aq = a.st.ahn + stash_tiled_off(cell, ntiles, tile, c, hs, 1, 0, 0) + 4 * row;
        const float *hq = a.st.h + stash_tiled_off(cell - (t > 0 ? 1 : 0), ntiles, tile, c, hs, 1, 0, 0) + 4 * row;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          sr[i] = __ldg(reinterpret_cast<const float4 *>(gq + i * 256));
          su[i] = __ldg(reinterpret_cast<const float4 *>(gq + 1024 + i * 256));
          sn[i] = __ldg(reinterpret_cast<const float4 *>(gq + 2048 + i * 256));
          sa[i] = __ldg(reinterpret_cast<const float4 *>(aq + i * 256));
          sh[i] = t > 0 ? __ldg(reinterpret_cast<const float4 *>(hq + i * 256)) : make_float4(0.f, 0.f, 0.f, 0.f);
          if (!rowok) sr[i] = su[i] = sn[i] = sa[i] = sh[i] = make_float4(0.f, 0.f, 0.f, 0.f);  // tile padding: no NaN from stale memory
        }
      }
      if (t < Tp - 1) {  // the peer's share of d h[k][t] (it rewrites this buffer only after X2 of this frame)
        const float *hp = dhc + (hs * PR + row) * 16;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 v = *reinterpret_cast<const float4 *>(hp + 4 * i);
          carry[4 * i] += v.x; carry[4 * i + 1] += v.y; carry[4 * i + 2] += v.z; carry[4 * i + 3] += v.w;
        }
      }
      // ---- 3. dh = dlin @ Wf (tensor cores) + carried gradient; 4. GRU gate backward --------------------------------------
      float dar[16], dau[16], dan[16], dnr[16];
      {
        mbar_wait(bar1, ph);
        fence_after();
        float lz[16];
        tmem_ld16(tlane + kColLZ + half * 32 + 16 * sub, lz);
        tmem_ld_wait();
        TSTAMPT(3);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float rg4[4] = {sr[i].x, sr[i].y, sr[i].z, sr[i].w}, ug4[4] = {su[i].x, su[i].y, su[i].z, su[i].w};
          const float ng4[4] = {sn[i].x, sn[i].y, sn[i].z, sn[i].w}, an4[4] = {sa[i].x, sa[i].y, sa[i].z, sa[i].w};
          const float hp4[4] = {sh[i].x, sh[i].y, sh[i].z, sh[i].w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int j = 4 * i + e;
            const float g = rowok ? carry[j] + lz[j] : 0.f;
            const float rgt = rg4[e], ug = ug4[e], ng = ng4[e];
            const float dn = g * (1.0f - ug), du = g * (hp4[e] - ng);
            const float v_an = dn * (1.0f - ng * ng);
            dan[j] = v_an;
            dau[j] = du * ug * (1.0f - ug);
            dar[j] = v_an * an4[e] * rgt * (1.0f - rgt);
            dnr[j] = v_an * rgt;
            carry[j] = g * ug;
          }
        }
      }
      // gate gradients as operand planes: shared memory (k-blocks r, u, n of this sequence) and the global dG / dA_h planes
      uint4 rh0, rl0, rh1, rl1, uh0, ul0, uh1, ul1, nh0, nl0, nh1, nl1, qh0, ql0, qh1, ql1;
      {
        auto split16 = [](const float (&v)[16], uint4 &h0, uint4 &l0, uint4 &h1, uint4 &l1) {
          const float a0[8] = {v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]}, a1[8] = {v[8], v[9], v[10], v[11], v[12], v[13], v[14], v[15]};
          split8(a0, h0, l0);
          split8(a1, h1, l1);
        };
        split16(dar, rh0, rl0, rh1, rl1);
        split16(dau, uh0, ul0, uh1, ul1);
        split16(dan, nh0, nl0, nh1, nl1);
        split16(dnr, qh0, ql0, qh1, ql1);
        const uint32_t o0 = kADA + sw128_off(row, ub >> 3), o1 = kADA + sw128_off(row, (ub >> 3) + 1);
        *reinterpret_cast<uint4 *>(smb + o0) = rh0; *reinterpret_cast<uint4 *>(smb + o0 + kADAPlane) = rl0;
        *reinterpret_cast<uint4 *>(smb + o1) = rh1; *reinterpret_cast<uint4 *>(smb + o1 + kADAPlane) = rl1;
        *reinterpret_cast<uint4 *>(smb + o0 + 64 * 128) = uh0; *reinterpret_cast<uint4 *>(smb + o0 + 64 * 128 + kADAPlane) = ul0;
        *reinterpret_cast<uint4 *>(smb + o1 + 64 * 128) = uh1; *reinterpret_cast<uint4 *>(smb + o1 + 64 * 128 + kADAPlane) = ul1;
        *reinterpret_cast<uint4 *>(smb + o0 + 2 * 64 * 128) = nh0; *reinterpret_cast<uint4 *>(smb + o0 + 2 * 64 * 128 + kADAPlane) = nl0;
        *reinterpret_cast<uint4 *>(smb + o1 + 2 * 64 * 128) = nh1; *reinterpret_cast<uint4 *>(smb + o1 + 2 * 64 * 128 + kADAPlane) = nl1;
      }
      fence_before();
      fence_async_smem();
      bar_arrive(2);  // the MMA warp issues P2 (dz1)
      TSTAMPT(4);
      // dA_i -> dG planes (time-parallel backward) straight from the shared-memory operand blocks: a block row holds the 64 units
      // of one gate = 128 contiguous bytes of the global row, so the copy is fully coalesced (8 lanes per row)
      auto copy_blocks = [&](void *ghi, void *glo, size_t row_base, size_t row_pitch, size_t col0, int blk_last) {
        // blocks 0, 1 and blk_last (2 = the n block as it is now) -> gate columns r, u, n of this CTA's units
        for (int e = tid; e < 3 * 64 * 8; e += PNT) {
          const int g = e >> 9, r = (e >> 3) & 63, ch = e & 7;
          if (r < nrows) {
            const uint32_t so = kADA + (uint32_t)(g == 2 ? blk_last : g) * (64 * 128) + sw128_off(r, ch);
            const size_t go = (row_base + r) * row_pitch + col0 + (size_t)g * H + 8 * ch;
            *reinterpret_cast<uint4 *>((__nv_bfloat16 *)ghi + go) = *reinterpret_cast<const uint4 *>(smb + so);
            if (glo) *reinterpret_cast<uint4 *>((__nv_bfloat16 *)glo + go) = *reinterpret_cast<const uint4 *>(smb + so + kADAPlane);
          }
        }
      };
      csync();  // every sequence's gate gradients are in the operand blocks
      if (a.pdG_hi) copy_blocks(a.pdG_hi, a.pdG_lo, (size_t)t * B + row0, (size_t)K * GH, (size_t)k * GH + PUC * c, 2);
      // ---- 5a. dz1 partial = dA_i W_ih[:, :Ci] (tensor cores): own rows into dzf, the peer's rows into its exchange buffer ----
      mbar_wait(bar2, ph);
      fence_after();
      if (q < 2) {  // lanes 0..63 hold the 64 sequences; the two warps of a quarter take 16 columns each
        float zv[16];
        tmem_ld16(tlane + kColZ + 16 * sub, zv);
        tmem_ld_wait();
        const int dest = row >> 5, lr = row & 31;
        if (dest == c) {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (16 * sub + j < Ci) dzf[lr * pC + 16 * sub + j] += zv[j];
        } else {
          float *ob = (float *)(peerb + pl.dz1x) + lr * 32 + 16 * sub;
#pragma unroll
          for (int i = 0; i < 4; ++i) *reinterpret_cast<float4 *>(ob + 4 * i) = make_float4(zv[4 * i], zv[4 * i + 1], zv[4 * i + 2], zv[4 * i + 3]);
        }
      }
      csync();  // the dG copy above has read the n block everywhere
      {  // n block of the gate gradients: d a_n -> r * d a_n for the recurrent product
        const uint32_t o0 = kADA + 2 * 64 * 128 + sw128_off(row, ub >> 3), o1 = kADA + 2 * 64 * 128 + sw128_off(row, (ub >> 3) + 1);
        *reinterpret_cast<uint4 *>(smb + o0) = qh0; *reinterpret_cast<uint4 *>(smb + o0 + kADAPlane) = ql0;
        *reinterpret_cast<uint4 *>(smb + o1) = qh1; *reinterpret_cast<uint4 *>(smb + o1 + kADAPlane) = ql1;
      }
      fence_before();
      fence_async_smem();
      bar_arrive(3);  // the MMA warp issues P3 (dh_prev)
      csync();        // the n block now holds r * d a_n for every sequence
      if (a.pdAh_hi) copy_blocks(a.pdAh_hi, a.pdAh_lo, cell * B + row0, (size_t)GH, (size_t)PUC * c, 2);  // dA_h planes (dW_hh)
      TSTAMPT(5);
      // ActNorm outputs for d logs of this thread's 1x1-conv-backward outputs, requested before the barrier
      float yv[2][4];
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int r = 2 * krp + i;
          yv[i][j] = (kact && r < nmy && 4 * kcq + j < C) ? __ldg(a.st.y + (cell * B + row0 + lr0 + r) * C + 4 * kcq + j) : 0.f;
        }
      cluster_arrive(); cluster_wait();  // X2: dz1 partial sums exchanged
      TSTAMPT(6);

      // ---- 6. finish d(1x1 conv output), dy = dzf @ W^T, ActNorm backward (modules.py:45-66) ------------------------------
      for (int e = tid; e < PRH * Ci; e += PNT) {
        const int r = fast_div(e, magCi), i = e - r * Ci;
        dzf[r * pC + i] += dz1x[r * 32 + i];
      }
      csync();
      if (kact) {
        float dy[2][4];
#pragma unroll
        for (int i = 0; i < 2; ++i) dy[i][0] = dy[i][1] = dy[i][2] = dy[i][3] = 0.f;
        const float *x0p = dzf + (2 * krp) * pC, *x1p = x0p + pC;
#pragma unroll 8
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
        csync();
        if (tid == 0) st_release_gpu_bt(my_flag, it + 1);  // release at gpu scope, cumulative over the barrier above
      }
      for (int e = tid; e < nmy * C; e += PNT) {  // dW (1x1 conv) operand stash: off the stage-to-stage path
        const int r = fast_div(e, magC), j = e - r * C;
        const size_t o = (cell * B + row0 + lr0 + r) * C + j;
        if (a.dzf) a.dzf[o] = dzf[r * pC + j];
        if (a.pdzf_hi) put_plane(a.pdzf_hi, a.pdzf_lo, o, dzf[r * pC + j]);
      }
      TSTAMPT(7);
      // ---- 5b. dh_prev partial = dA_h W_hh (tensor cores): own units -> carry, the peer's units -> its exchange buffer --------
      {
        mbar_wait(bar3, ph);
        fence_after();
        float own[16], oth[16];
        tmem_ld16(tlane + kColHP + half * 64 + 16 * sub, own);
        tmem_ld16(tlane + kColHP + half * 64 + 32 + 16 * sub, oth);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) carry[j] += own[j];
        float *pq = (float *)(peerb + pl.dhc) + (hs * PR + row) * 16;
#pragma unroll
        for (int i = 0; i < 4; ++i) *reinterpret_cast<float4 *>(pq + 4 * i) = make_float4(oth[4 * i], oth[4 * i + 1], oth[4 * i + 2], oth[4 * i + 3]);
        fence_before();
      }
      csync();  // every compute thread is done with dzf before the next frame's coupling rewrites it
      cluster_arrive();  // X3 (split): done with the operand blocks, the peer's dh_prev share delivered
      x3_pending = true;
      TSTAMPT(8);
    }
    if (x3_pending) { cluster_wait(); x3_pending = false; }
  }

  if (timing)
    printf("core_bwd_pipe_tc stage %d: frames %d cycles/frame: prefetch+wait %lld | coupling bwd+dlin planes %lld | X1 %lld | P1 wait %lld | gate bwd+planes %lld | dG/dAh stores, P2 wait, dz1 exchange %lld | X2 %lld | dzf, 1x1 bwd, publish, stash %lld | P3 wait+exchange %lld\n",
           k, it, tacc[0] / it, tacc[1] / it, tacc[2] / it, tacc[3] / it, tacc[4] / it, tacc[5] / it, tacc[6] / it, tacc[7] / it, tacc[8] / it);
  // ---- flush the per-channel gradients --------------------------------------------------------------------------------
  if (!mma_warp) {
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
  fence_before();
  __syncthreads();
  if (mma_warp) {
    fence_after();
    tmem_dealloc(tmem, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------
bool pipe_bwd_tc_supported(const Dims &d) { return plan_bt(d).total <= 227 * 1024; }

int launch_bwd_pipe_tc(const BwdArgs &a, cudaStream_t st) {
  LFI_REQUIRE(a.stash_tiled && a.pdG_hi && a.pdAh_hi, LFI_ERR_ARG, "tensor-core backward pipeline needs the tiled stash and plane outputs");
  static const int timing = getenv("LFI_CORE_TIMING") ? atoi(getenv("LFI_CORE_TIMING")) : 0;
  if (timing) cudaMemcpyToSymbolAsync(g_core_timing_bt, &timing, sizeof(int), 0, cudaMemcpyHostToDevice, st);
  auto kern = a.dx_in ? core_bwd_pipe_tc<true> : core_bwd_pipe_tc<false>;
  return launch_pipe(kern, a, BNT, plan_bt(a.d).total, a.d.K, a.d.K + 1, "core_bwd_pipe_tc", st);
}

}  // namespace core
}  // namespace lfi
