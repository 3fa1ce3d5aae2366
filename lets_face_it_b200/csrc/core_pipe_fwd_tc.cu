// Persistent stage-pipelined flow core, forward direction, gate products on the tensor cores (tensor-core GEMM modes).
//
// Same scheme as core_pipe_fwd.cu (one 2-CTA cluster per flow step, weights and RNN state resident in shared memory
// across all frames, stages chained by release/acquire counters), but the three products of the coupling network
//   h_{t-1} W_hh^T   [64 x 128] x [128 x 192]     (this CTA's 64 hidden units x r, u, n)
//   z1 W_ih[:, :Ci]^T [64 x 28]  x [28 x 192]
//   h_t Wf^T          [64 x 64]  x [64 x 56]       (LinearZeros, partial sum over this CTA's units)
// are tcgen05.mma instructions (fp32 accumulation in TMEM) on split-bf16 operands.  A tile has 64 sequences but the MMA has
// M = 128 accumulator lanes: every product is issued twice, once on the A operand as stored (sequences in lanes 0..63)
// against the weight rows of hidden units 0..31, once with the A descriptor moved back by 64 rows (the same sequences
// land in lanes 64..127) against the rows of units 32..63 - all 128 lanes, i.e. all eight warps, then hold useful
// accumulators (thread = sequence x 16 hidden units).  Operands: a = a_hi + a_lo, three products a_hi b_hi + a_hi b_lo +
// a_lo b_hi, fp32-grade (same numerics as the bf16x3 GEMMs of the time-parallel phase).  A ninth warp issues every MMA, so
// that the issue latency of the frame's ~100 instructions never holds up the eight compute warps (they synchronise among
// themselves with a named barrier and with the issuer through bar.arrive / bar.sync and mbarrier commits).  The weights are split once per launch into resident hi / lo planes in the canonical
// K-major swizzled UMMA layout; the state h and z1 are written as hi / lo planes by the threads that produce them (own
// half locally, the other CTA's copy through distributed shared memory).  Gate math reads the accumulators with
// tcgen05.ld (thread = sequence) - reference: nn.GRUCell inside f_seq.forward, models.py:204-214; LinearZeros
// modules.py:83-95.
#include "core_pipe.cuh"
#include "tc_ptx.cuh"
#include <cooperative_groups.h>
#include <cstdlib>

namespace cg = cooperative_groups;

namespace lfi {
namespace core {

using namespace tcp;

namespace {

__device__ __forceinline__ int ld_acquire_gpu_t(const int *p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu_t(int *p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}

constexpr int FNT = 288;  // eight compute warps + the MMA-issue warp
__device__ __forceinline__ void csync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }  // the eight compute warps
__device__ __forceinline__ bool csync_and(bool pred) {
  uint32_t r;
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "setp.ne.u32 q, %1, 0;\n\t"
      "bar.red.and.pred p, 1, 256, q;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(r) : "r"((uint32_t)pred) : "memory");
  return r != 0;
}
__device__ __forceinline__ void bar_arrive2() { asm volatile("bar.arrive 2, 288;" ::: "memory"); }
__device__ __forceinline__ void cluster_arrive_() { asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory"); }
__device__ __forceinline__ void cluster_wait_() { asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory"); }
__device__ __forceinline__ void bar_sync2() { asm volatile("bar.sync 2, 288;" ::: "memory"); }

// byte offsets of the operand blocks (all 1024-byte aligned)
constexpr int kBH = 0;                  // W_hh slice   2 planes x 2 k-blocks x [192 rows x 128 B]   (128-byte swizzle)
constexpr int kBHPlane = 2 * 192 * 128; //   48 KB per plane, 24 KB per k-block
constexpr int kBZ = kBH + 2 * kBHPlane; // W_ih[:, :Ci] 2 planes x [192 rows x 64 B]                 (64-byte swizzle)
constexpr int kBZPlane = 192 * 64;
constexpr int kBF = kBZ + 2 * kBZPlane; // Wf slice     2 planes x [64 rows x 128 B]                 (128-byte swizzle)
constexpr int kBFPlane = 64 * 128;
constexpr int kAH = kBF + 2 * kBFPlane; // h            2 planes x 2 k-blocks x [64 rows x 128 B]
constexpr int kAHPlane = 2 * 64 * 128;  //   the MMA (M = 128) reads 128 rows per k-block: rows 64.. alias the bytes that follow
constexpr int kAZ = kAH + 2 * kAHPlane; // z1           2 planes x [64 rows x 64 B]
constexpr int kAZPlane = 64 * 64;
constexpr int kF32 = kAZ + 2 * kAZPlane;  // fp32 arrays follow (they also back the aliased rows of the last A block)
constexpr int kTmemCols = 512;
constexpr int kColD = 0, kColF = 256;   // accumulators: [0,64) r, [64,128) u, [128,192) n (h side), [192,256) n (i side); LinearZeros
__device__ int g_core_timing = 0;  // debug: LFI_CORE_TIMING=1 prints the phase cycle counts of one CTA

struct PlanTC {
  int w, vec, xs, zrow, o, bars, total;  // byte offsets
  int pC, pO;
};
__host__ __device__ inline PlanTC plan_tc(const Dims &d) {
  PlanTC p;
  p.pC = odd(d.C);
  p.pO = round_up(d.Co, 4) + 4;
  int o = kF32;
  auto take = [&](int nfloats) { int r = o; o += round_up(nfloats, 4) * 4; return r; };
  p.w = take(d.C * d.Cp);
  p.vec = take(2 * d.C + 3 * PUC + 2 * d.Co);
  p.xs = take(PRH * p.pC);
  p.zrow = take(PRH * p.pC);
  p.o = take(2 * PRH * p.pO);
  p.bars = take(16);
  p.total = o + 1024;  // alignment reserve
  return p;
}

}  // namespace

// kCarry: every tile starts from the state a.h0 [K][B][H] and leaves its last frame's state in a.h_last [K][B][H] (time-chunked
// evaluation, lfi_seq_eval); there is no st_h stash.  The instantiation without it starts from zeros and stores st_h.
template <bool kCarry>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(FNT, 1)
core_fwd_pipe_tc(const FwdArgs a, const int P, const int ntiles, int *progress) {
  extern __shared__ __align__(16) uint8_t smraw[];
  uint8_t *smb = (uint8_t *)(((uintptr_t)smraw + 1023) & ~(uintptr_t)1023);
  cg::cluster_group cluster = cg::this_cluster();
  const Dims &d = a.d;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = (int)cluster.block_rank();
  const int stage = blockIdx.y, nk = gridDim.y, k = a.k_first + stage, p = blockIdx.z;
  const int C = d.C, Ci = d.Ci, Cz = d.Cz, Co = d.Co, H = d.H, GH = d.GH, B = a.B, Tp = a.Tp, Cp = d.Cp, Cip = d.Cip;
  const unsigned magC = div_magic(C);
  const PlanTC pl = plan_tc(d);
  const int pC = pl.pC, pO = pl.pO;
  float *wsm = (float *)(smb + pl.w);
  float *anb = (float *)(smb + pl.vec), *ans = anb + C, *bhh = ans + C, *bfs = bhh + 3 * PUC, *e3 = bfs + Co;
  float *xs = (float *)(smb + pl.xs), *zrow = (float *)(smb + pl.zrow), *osm = (float *)(smb + pl.o);
  uint64_t *bar_hh = (uint64_t *)(smb + pl.bars), *bar_d = bar_hh + 1, *bar_f = bar_hh + 2;
  uint32_t *tmem_slot = (uint32_t *)(bar_hh + 3);
  uint8_t *peerb = cluster.map_shared_rank(smb, c ^ 1);
  const StepWeights w = a.dv.step(d, k);
  const bool first = (k == a.k_first), last = (k == a.k_last);

  // ---- resident weights: fp32 -> (hi, lo) bf16 planes in the K-major swizzled UMMA layout ------------------------
  for (int e = tid; e < 192 * 16; e += FNT) {  // W_hh[g*H + 64c + u][8ch .. 8ch+7]
    const int n = e >> 4, ch = e & 15, g = n >> 6, u = n & 63;
    const float *src = w.Whh + (size_t)(g * H + PUC * c + u) * H + 8 * ch;
    const float4 v0 = *reinterpret_cast<const float4 *>(src), v1 = *reinterpret_cast<const float4 *>(src + 4);
    const float v[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
    uint4 hi, lo;
    split8(v, hi, lo);
    const int np = (u >> 5) * 96 + g * 32 + (u & 31);  // rows grouped by unit half: [half][gate][32 units]
    const uint32_t off = (uint32_t)(ch >> 3) * (192 * 128) + sw128_off(np, ch & 7);
    *reinterpret_cast<uint4 *>(smb + kBH + off) = hi;
    *reinterpret_cast<uint4 *>(smb + kBH + kBHPlane + off) = lo;
  }
  for (int e = tid; e < 192 * 4; e += FNT) {   // W_ih[g*H + 64c + u][8ch .. 8ch+7], zero beyond Ci
    const int n = e >> 2, ch = e & 3, g = n >> 6, u = n & 63;
    const float *src = w.WihZ + (size_t)(g * H + PUC * c + u) * Cip;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = (8 * ch + j < Ci) ? src[8 * ch + j] : 0.f;
    uint4 hi, lo;
    split8(v, hi, lo);
    const int np = (u >> 5) * 96 + g * 32 + (u & 31);
    const uint32_t off = sw64_off(np, ch);
    *reinterpret_cast<uint4 *>(smb + kBZ + off) = hi;
    *reinterpret_cast<uint4 *>(smb + kBZ + kBZPlane + off) = lo;
  }
  for (int e = tid; e < 64 * 8; e += FNT) {    // Wf[j][64c + 8ch .. +7], zero rows beyond Co
    const int n = e >> 3, ch = e & 7;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = (n < Co) ? w.Wf[(size_t)n * H + PUC * c + 8 * ch + j] : 0.f;
    uint4 hi, lo;
    split8(v, hi, lo);
    const uint32_t off = sw128_off(n, ch);
    *reinterpret_cast<uint4 *>(smb + kBF + off) = hi;
    *reinterpret_cast<uint4 *>(smb + kBF + kBFPlane + off) = lo;
  }
  for (int e = tid; e < C * (Cp / 4); e += FNT)
    *reinterpret_cast<float4 *>(wsm + 4 * e) = *reinterpret_cast<const float4 *>(w.Wfwd + 4 * e);
  for (int e = tid; e < C; e += FNT) { anb[e] = w.an_bias[e]; ans[e] = expf(w.an_logs[e]); }
  for (int e = tid; e < 3 * PUC; e += FNT) bhh[e] = w.b_hh[(e / PUC) * H + PUC * c + (e % PUC)];
  for (int e = tid; e < Co; e += FNT) { bfs[e] = w.bf[e]; e3[e] = expf(3.0f * w.lf[e]); }
  for (int e = tid; e < 2 * kAZPlane / 16; e += FNT) reinterpret_cast<uint4 *>(smb + kAZ)[e] = make_uint4(0u, 0u, 0u, 0u);
  if (tid == 0) {
    mbar_init(bar_hh, 1); mbar_init(bar_d, 1); mbar_init(bar_f, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  const bool mma_warp = warp == 8;
  if (mma_warp) tmem_alloc(tmem_slot, kTmemCols);
  fence_before();
  fence_async_smem();
  cluster.sync();  // both CTAs of the cluster are running before the first distributed-shared-memory access
  fence_after();
  const uint32_t tmem = *tmem_slot;

  // accumulators: TMEM lane L = 32 (warp % 4) + lane holds sequence L % 64 of the tile and the hidden units of half L / 64;
  // the two warps of a lane quarter split that half's 32 units
  const int q = warp & 3, sub = warp >> 2;
  const int L = 32 * q + lane, row = L & 63, half = q >> 1;
  const int ub = 32 * half + 16 * sub;  // first of this thread's 16 hidden units (inside the CTA's 64)
  const uint32_t tlane = tmem + ((uint32_t)(32 * q) << 16);
  const uint32_t colR = kColD + half * 96 + 16 * sub, colU = colR + 32, colH = colR + 64, colI = kColD + 192 + half * 32 + 16 * sub;
  const int lr0 = PRH * c;  // first tile row of this CTA's row half
  const int *wait_flag = progress + ((size_t)(p * nk + stage - 1) * 2 + c);
  int *my_flag = progress + ((size_t)(p * nk + stage) * 2 + c);
  const uint32_t sAH = smem_u32(smb + kAH), sAZ = smem_u32(smb + kAZ), sBH = smem_u32(smb + kBH), sBZ = smem_u32(smb + kBZ),
                 sBF = smem_u32(smb + kBF);
  int it = 0;
  const bool timing = g_core_timing && tid == 0 && c == 0 && p == 0 && (stage == 8 || stage == 0 || stage == nk - 1);
  long long tacc[20] = {0}, tprev = 0;
#define TSTAMP(i) do { if (timing) { const long long now_ = clock64(); tacc[i] += now_ - tprev; tprev = now_; } } while (0)

  for (int tile = p; tile < ntiles; tile += P) {
    const int row0 = tile * PR, nrows = min(PR, B - row0);
    const int nmy = max(0, min(PRH, nrows - lr0));
    float hreg[16];
    if constexpr (kCarry) {
      // the carried state of this thread's sequence and 16 units, as operand planes of this CTA's k-block in both CTAs (the
      // per-frame update's layout); rows past the batch are zero.  The compute threads of the two CTAs together write both
      // k-blocks whole, so nothing is zeroed first.
      if (!mma_warp) {
        const bool ok = row < nrows;
        const float *src = a.h0 + ((size_t)k * B + row0 + row) * H + PUC * c + ub;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 v = ok ? *reinterpret_cast<const float4 *>(src + 4 * i) : make_float4(0.f, 0.f, 0.f, 0.f);
          hreg[4 * i] = v.x; hreg[4 * i + 1] = v.y; hreg[4 * i + 2] = v.z; hreg[4 * i + 3] = v.w;
        }
        uint4 hi0, lo0, hi1, lo1;
        {
          const float v0[8] = {hreg[0], hreg[1], hreg[2], hreg[3], hreg[4], hreg[5], hreg[6], hreg[7]};
          const float v1[8] = {hreg[8], hreg[9], hreg[10], hreg[11], hreg[12], hreg[13], hreg[14], hreg[15]};
          split8(v0, hi0, lo0);
          split8(v1, hi1, lo1);
        }
        const uint32_t o0 = kAH + (uint32_t)c * (64 * 128) + sw128_off(row, ub >> 3), o1 = kAH + (uint32_t)c * (64 * 128) + sw128_off(row, (ub >> 3) + 1);
        *reinterpret_cast<uint4 *>(smb + o0) = hi0; *reinterpret_cast<uint4 *>(smb + o0 + kAHPlane) = lo0;
        *reinterpret_cast<uint4 *>(smb + o1) = hi1; *reinterpret_cast<uint4 *>(smb + o1 + kAHPlane) = lo1;
        *reinterpret_cast<uint4 *>(peerb + o0) = hi0; *reinterpret_cast<uint4 *>(peerb + o0 + kAHPlane) = lo0;
        *reinterpret_cast<uint4 *>(peerb + o1) = hi1; *reinterpret_cast<uint4 *>(peerb + o1 + kAHPlane) = lo1;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j) hreg[j] = 0.f;
      for (int e = tid; e < 2 * kAHPlane / 16; e += FNT) reinterpret_cast<uint4 *>(smb + kAH)[e] = make_uint4(0u, 0u, 0u, 0u);  // state None = zeros
    }
    fence_async_smem();
    cluster.sync();

    for (int t = 0; t < Tp; ++t, ++it) {
      const size_t cell = (size_t)k * Tp + t;
      const uint32_t ph = (uint32_t)(it & 1);
      if (mma_warp) {
        // =================================== MMA-issue warp ===================================
        if (lane == 0) {  // recurrent product h_{t-1} W_hh^T: no dependence on stage k-1, overlaps the wait for it

        fence_after();
        fence_async_smem();
        const uint32_t idesc = idesc_bf16_m128(96);
        uint32_t acc = 0;
#pragma unroll
        for (int pr = 0; pr < 3; ++pr) {  // (hi,hi), (hi,lo), (lo,hi)
          const uint32_t pa = (pr == 2) ? kAHPlane : 0, pb = (pr == 1) ? kBHPlane : 0;
#pragma unroll
          for (int kb = 0; kb < 2; ++kb)
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
              for (int hf = 0; hf < 2; ++hf)  // hf = 1: A moved back by 64 rows, weight rows of units 32..63
                umma_bf16(tmem + kColD + hf * 96, make_sdesc(sAH + pa + kb * (64 * 128) + ks * 32 - hf * (64 * 128), 1024, kSw128),
                          make_sdesc(sBH + pb + kb * (192 * 128) + hf * (96 * 128) + ks * 32, 1024, kSw128), idesc, acc);
              acc = 1;
            }
        }
        umma_commit(bar_hh);
              }
        __syncwarp();
        mbar_wait(bar_hh, ph);  // this CTA's recurrent product has consumed h_{t-1}: the peer may overwrite its half after A
        cluster_arrive_(); cluster_wait_();  // A: z1 complete in both CTAs
        if (lane == 0) {

        fence_after();
        fence_async_smem();
        const uint32_t id_ru = idesc_bf16_m128(64), id_n = idesc_bf16_m128(32);
        uint32_t accn = 0;
#pragma unroll
        for (int pr = 0; pr < 3; ++pr) {
          const uint32_t pa = (pr == 2) ? kAZPlane : 0, pb = (pr == 1) ? kBZPlane : 0;
#pragma unroll
          for (int ks = 0; ks < 2; ++ks) {
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
              const uint64_t ad = make_sdesc(sAZ + pa + ks * 32 - hf * (64 * 64), 512, kSw64);
              const uint32_t sb = sBZ + pb + hf * (96 * 64) + ks * 32;
              umma_bf16(tmem + kColD + hf * 96, ad, make_sdesc(sb, 512, kSw64), id_ru, 1u);                        // r, u
              umma_bf16(tmem + kColD + 192 + hf * 32, ad, make_sdesc(sb + 64 * 64, 512, kSw64), id_n, accn);     // n, input side
            }
            accn = 1;
          }
        }
        umma_commit(bar_d);
              }
        __syncwarp();
        bar_sync2();  // gate math done: the new state is in the operand planes
        if (lane == 0) {

        fence_after();
        fence_async_smem();
        const uint32_t idesc = idesc_bf16_m128(32);
        uint32_t acc = 0;
#pragma unroll
        for (int pr = 0; pr < 3; ++pr) {
          const uint32_t pa = (pr == 2) ? kAHPlane : 0, pb = (pr == 1) ? kBFPlane : 0;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
            for (int hf = 0; hf < 2; ++hf)  // output channels 0..31 in lanes 0..63, channels 32..63 in lanes 64..127
              umma_bf16(tmem + kColF + hf * 32, make_sdesc(sAH + pa + c * (64 * 128) + ks * 32 - hf * (64 * 128), 1024, kSw128),
                        make_sdesc(sBF + pb + hf * (32 * 128) + ks * 32, 1024, kSw128), idesc, acc);
            acc = 1;
          }
        }
        umma_commit(bar_f);
              }
        __syncwarp();
        cluster_arrive_(); cluster_wait_();  // B
        continue;
      }
      if (timing) tprev = clock64();
      //         request the input if stage k-1 has already published this frame (it usually runs ahead)
      constexpr int XI = (PRH * 64 + PNT - 1) / PNT;  // C <= 64
      float xv[XI];
      bool have_x = first || ld_acquire_gpu_t(wait_flag) > it;
      have_x = csync_and(have_x);
      TSTAMP(0);
      auto fetch_x = [&]() {
#pragma unroll
        for (int i = 0; i < XI; ++i) {
          const int e = tid + PNT * i, r = fast_div(e, magC), cc = e - r * C;
          xv[i] = 0.f;
          if (e < PRH * C && r < nmy) {
            const int b = row0 + lr0 + r;
            xv[i] = first ? a.x0[(size_t)b * a.x_sb + (size_t)t * a.x_st + cc] : __ldcg(a.xin + (cell * B + b) * C + cc);
          }
        }
      };
      if (have_x) fetch_x();

      // ---- 1. wait for stage k-1, ActNorm (modules.py:45-66) on this CTA's 32 rows ---------------------------------
      if (!have_x) {
        if (tid == 0) {
          spin_wait_gt(wait_flag, it);
        }
        csync();
        fetch_x();
      }
#pragma unroll
      for (int i = 0; i < XI; ++i) {
        const int e = tid + PNT * i, r = fast_div(e, magC), cc = e - r * C;
        if (e < PRH * C) {
          float v = 0.f;
          if (r < nmy) {
            v = (xv[i] + anb[cc]) * ans[cc];
          }
          xs[r * pC + cc] = v;
        }
      }
      csync();
      TSTAMP(1);
      // ---- 2. invertible 1x1 conv (modules.py:186): z = y @ W, 2 rows x 4 columns per thread (fp32 FFMA) -----------
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
#pragma unroll 8
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
      csync();
      TSTAMP(2);
      if (tid < PRH * 4) {  // z1 of this CTA's rows as operand planes, to both CTAs of the cluster
        const int r = tid >> 2, ch = tid & 3;
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = (8 * ch + j < Ci) ? zrow[r * pC + 8 * ch + j] : 0.f;
        uint4 hi, lo;
        split8(v, hi, lo);
        const uint32_t off = kAZ + sw64_off(lr0 + r, ch);
        *reinterpret_cast<uint4 *>(smb + off) = hi;
        *reinterpret_cast<uint4 *>(smb + off + kAZPlane) = lo;
        *reinterpret_cast<uint4 *>(peerb + off) = hi;
        *reinterpret_cast<uint4 *>(peerb + off + kAZPlane) = lo;
      }
      fence_async_smem();
      cluster_arrive_();  // A: z1 complete in both CTAs (the MMA warp joins once its recurrent product is done)
      for (int e = tid; e < nmy * C; e += PNT) {  // y stash of this CTA's rows (fp32 and operand planes) inside the barrier window
        const int r = fast_div(e, magC), j = e - r * C;
        const size_t o = (cell * B + row0 + lr0 + r) * C + j;
        const float yv = xs[r * pC + j];
        if (a.st_y) a.st_y[o] = yv;
        if (a.py_hi) put_plane(a.py_hi, a.py_lo, o, yv);
      }
      cluster_wait_();
      TSTAMP(3);
      // ---- 3. z1 part of the gate-ih product, then the GRU gate math straight from TMEM -------------------------------
      //         gate-ih pre-activations of the first pass (requested here: their issue overlaps the z1 product)
      const size_t gm = (size_t)t * B + row0 + row, gn = (size_t)(k - a.g_k0) * GH + PUC * c + ub;
      const float *Gb = a.g_tiled ? a.G + g_tiled_off(gm, gn, (size_t)a.g_ld) : a.G + gm * a.g_ld + gn;
      const size_t gstep_g = a.g_tiled ? (size_t)(H >> 2) * 128 : (size_t)H, gstep_i = a.g_tiled ? 128 : 4;  // next gate / next 4 columns
      const bool rowok = row < nrows;
      float4 gq[3][4];
#pragma unroll
      for (int g = 0; g < 3; ++g)
#pragma unroll
        for (int i = 0; i < 4; ++i) gq[g][i] = rowok ? __ldg(reinterpret_cast<const float4 *>(Gb + g * gstep_g + i * gstep_i)) : make_float4(0.f, 0.f, 0.f, 0.f);
      float vr[16], vu[16], vh[16], vi[16];
      uint4 hi0, lo0, hi1, lo1;
      {
        mbar_wait(bar_d, ph);
        fence_after();
        TSTAMP(4);
        tmem_ld16(tlane + colR, vr);
        tmem_ld16(tlane + colU, vu);
        tmem_ld16(tlane + colH, vh);
        tmem_ld16(tlane + colI, vi);
        tmem_ld_wait();
        float hn[16];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float gr[4] = {gq[0][i].x, gq[0][i].y, gq[0][i].z, gq[0][i].w}, gu[4] = {gq[1][i].x, gq[1][i].y, gq[1][i].z, gq[1][i].w},
                      gi[4] = {gq[2][i].x, gq[2][i].y, gq[2][i].z, gq[2][i].w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int j = 4 * i + e;
            const float rgt = fast_sigmoid(vr[j] + gr[e] + bhh[ub + j]);
            const float ugt = fast_sigmoid(vu[j] + gu[e] + bhh[PUC + ub + j]);
            const float anh = vh[j] + bhh[2 * PUC + ub + j];
            const float ng = fast_tanh(vi[j] + gi[e] + rgt * anh);
            vr[j] = rgt; vu[j] = ugt; vh[j] = anh; vi[j] = ng;
            hn[j] = ng + ugt * (hreg[j] - ng);
            hreg[j] = hn[j];
          }
        }
        // new state as operand planes: own k-block (hidden units 64c ..) of h in both CTAs, and the global planes
        {
          const float v0[8] = {hn[0], hn[1], hn[2], hn[3], hn[4], hn[5], hn[6], hn[7]};
          const float v1[8] = {hn[8], hn[9], hn[10], hn[11], hn[12], hn[13], hn[14], hn[15]};
          split8(v0, hi0, lo0);
          split8(v1, hi1, lo1);
        }
        {
          const uint32_t o0 = kAH + (uint32_t)c * (64 * 128) + sw128_off(row, ub >> 3), o1 = kAH + (uint32_t)c * (64 * 128) + sw128_off(row, (ub >> 3) + 1);
          *reinterpret_cast<uint4 *>(smb + o0) = hi0; *reinterpret_cast<uint4 *>(smb + o0 + kAHPlane) = lo0;
          *reinterpret_cast<uint4 *>(smb + o1) = hi1; *reinterpret_cast<uint4 *>(smb + o1 + kAHPlane) = lo1;
          *reinterpret_cast<uint4 *>(peerb + o0) = hi0; *reinterpret_cast<uint4 *>(peerb + o0 + kAHPlane) = lo0;
          *reinterpret_cast<uint4 *>(peerb + o1) = hi1; *reinterpret_cast<uint4 *>(peerb + o1 + kAHPlane) = lo1;
        }
        fence_before();      // this warp's accumulator reads are complete before the next products overwrite them
        fence_async_smem();  // the new state is visible to the tensor cores (of both CTAs)
        TSTAMP(5);
      }
      bar_arrive2();  // the MMA warp issues the LinearZeros product
      TSTAMP(6);

      // ---- 4. LinearZeros (modules.py:93-95): partial sum over this CTA's 64 hidden units, all 64 rows ---------------
      {  // stash for the backward pass (gates post-activation, h-side n pre-activation, new state) while it runs: tiled
         // layout, the 32 sequences of a warp are contiguous in every store (rows beyond the batch land in the tile's padding)
        const int hs = 2 * half + sub;
        if (a.st_gates) {
          float *gp = a.st_gates + stash_tiled_off(cell, ntiles, tile, c, hs, 3, 0, 0) + 4 * row;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            *reinterpret_cast<float4 *>(gp + i * 256) = make_float4(vr[4 * i], vr[4 * i + 1], vr[4 * i + 2], vr[4 * i + 3]);
            *reinterpret_cast<float4 *>(gp + 1024 + i * 256) = make_float4(vu[4 * i], vu[4 * i + 1], vu[4 * i + 2], vu[4 * i + 3]);
            *reinterpret_cast<float4 *>(gp + 2048 + i * 256) = make_float4(vi[4 * i], vi[4 * i + 1], vi[4 * i + 2], vi[4 * i + 3]);
          }
        }
      }
      {
        mbar_wait(bar_f, ph);
        fence_after();
        float ov[16];
        tmem_ld16(tlane + kColF + half * 32 + 16 * sub, ov);
        tmem_ld_wait();
        const int dest = row >> 5, lr = row & 31;  // CTA that owns this row; slot c holds this CTA's partial
        const int j0 = 32 * half + 16 * sub;
        float *ob = (float *)((dest == c ? smb : peerb) + pl.o) + c * PRH * pO + lr * pO + j0;
        const int Cop = d.Cop;
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (j0 + 4 * i < Cop) *reinterpret_cast<float4 *>(ob + 4 * i) = make_float4(ov[4 * i], ov[4 * i + 1], ov[4 * i + 2], ov[4 * i + 3]);
        fence_before();
      }
      cluster_arrive_();  // B: partial sums and the new state are complete in both CTAs
      {  // rest of the backward stash (h-side n pre-activation, new state, operand planes, zf) inside the barrier window
        const int hs = 2 * half + sub;
        if (a.st_ahn) {
          float *ap = a.st_ahn + stash_tiled_off(cell, ntiles, tile, c, hs, 1, 0, 0) + 4 * row;
#pragma unroll
          for (int i = 0; i < 4; ++i) *reinterpret_cast<float4 *>(ap + i * 256) = make_float4(vh[4 * i], vh[4 * i + 1], vh[4 * i + 2], vh[4 * i + 3]);
        }
        if constexpr (kCarry) {
          if (t == Tp - 1 && rowok) {
            float *hp = a.h_last + ((size_t)k * B + row0 + row) * H + PUC * c + ub;
#pragma unroll
            for (int i = 0; i < 4; ++i) *reinterpret_cast<float4 *>(hp + 4 * i) = make_float4(hreg[4 * i], hreg[4 * i + 1], hreg[4 * i + 2], hreg[4 * i + 3]);
          }
        } else {
          float *hp = a.st_h + stash_tiled_off(cell, ntiles, tile, c, hs, 1, 0, 0) + 4 * row;
#pragma unroll
          for (int i = 0; i < 4; ++i) *reinterpret_cast<float4 *>(hp + i * 256) = make_float4(hreg[4 * i], hreg[4 * i + 1], hreg[4 * i + 2], hreg[4 * i + 3]);
        }
        if (rowok && a.ph_hi) {
          const size_t rb = cell * B + row0 + row;
          const int uo = PUC * c + ub;
          __nv_bfloat16 *phi = (__nv_bfloat16 *)a.ph_hi + rb * H + uo;
          *reinterpret_cast<uint4 *>(phi) = hi0; *reinterpret_cast<uint4 *>(phi + 8) = hi1;
          if (a.ph_lo) {
            __nv_bfloat16 *plo = (__nv_bfloat16 *)a.ph_lo + rb * H + uo;
            *reinterpret_cast<uint4 *>(plo) = lo0; *reinterpret_cast<uint4 *>(plo + 8) = lo1;
          }
        }
      }
      for (int e = tid; e < nmy * C; e += PNT) {  // zf stash of this CTA's rows (fp32 and operand planes) 
        const int r = fast_div(e, magC), j = e - r * C;
        const size_t o = (cell * B + row0 + lr0 + r) * C + j;
        const float zv = zrow[r * pC + j];
        if (a.st_zf) a.st_zf[o] = zv;
        if (a.pzf_hi) put_plane(a.pzf_hi, a.pzf_lo, o, zv);
      }
      cluster_wait_();
      TSTAMP(7);

      // ---- 5. affine coupling (models.py:331-341), log-det, NLL on the last step (modules.py:207-212, models.py:563-565)
      //         a warp owns rows warp, warp + 8, ... of this CTA's 32; their chains are independent and interleaved
      {
        const float *o0 = osm, *o1 = osm + PRH * pO;
        constexpr int NRW = PRH / (PNT / 32);
        float ldv = 0.f;  // running log-det of row warp + 8 * lane: one round trip for the warp's rows
        if ((!first || a.ld_accumulate) && warp + (PNT / 32) * lane < nmy)
          ldv = __ldcg(a.ld + (size_t)t * B + row0 + lr0 + warp + (PNT / 32) * lane);
        float lsum[NRW], zsq[NRW];
#pragma unroll
        for (int n = 0; n < NRW; ++n) {
          const int r = warp + (PNT / 32) * n;
          lsum[n] = 0.f; zsq[n] = 0.f;
          if (r < nmy && lane < Cz) {
            const int b = row0 + lr0 + r, qq = lane;
            const float z2 = zrow[r * pC + Ci + qq];
            float znew;
            if (d.affine) {
              const float shift = (o0[r * pO + 2 * qq] + o1[r * pO + 2 * qq] + bfs[2 * qq]) * e3[2 * qq];
              const float sc = (o0[r * pO + 2 * qq + 1] + o1[r * pO + 2 * qq + 1] + bfs[2 * qq + 1]) * e3[2 * qq + 1];
              const float sg = fmaxf(fast_sigmoid(sc + 2.0f), d.eps);
              znew = (z2 + shift) * sg;
              lsum[n] = __logf(sg);
              if (a.st_o) *reinterpret_cast<float2 *>(a.st_o + (cell * B + b) * Co + 2 * qq) = make_float2(shift, sc);
              if (a.scale_out && t == Tp - 1) a.scale_out[((size_t)k * B + b) * Cz + qq] = sg;
            } else {
              const float ov = (o0[r * pO + qq] + o1[r * pO + qq] + bfs[qq]) * e3[qq];
              znew = z2 + ov;
              if (a.st_o) a.st_o[(cell * B + b) * Co + qq] = ov;
            }
            zrow[r * pC + Ci + qq] = znew;
            zsq[n] = znew * znew;
          }
          if (last && a.nll && r < nmy && lane < Ci) { const float z1v = zrow[r * pC + lane]; zsq[n] += z1v * z1v; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
          for (int n = 0; n < NRW; ++n) {
            lsum[n] += __shfl_xor_sync(0xffffffffu, lsum[n], o);
            zsq[n] += __shfl_xor_sync(0xffffffffu, zsq[n], o);
          }
#pragma unroll
        for (int n = 0; n < NRW; ++n) {
          const int r = warp + (PNT / 32) * n;
          const float ld = lsum[n] + __shfl_sync(0xffffffffu, ldv, n);
          if (r < nmy && lane == 0) {
            const int b = row0 + lr0 + r;
            if (last && a.nll) a.nll[(size_t)t * B + b] = -(ld - 0.5f * (zsq[n] + (float)C * kLog2Pi)) / kLn2;
            a.ld[(size_t)t * B + b] = ld;
          }
        }
      }
      csync();
      {
        float *dst = last ? a.z_out + (size_t)t * B * C : a.xin + (cell + Tp) * B * C;  // XIN[k+1][t]
        for (int e = tid; e < nmy * C; e += PNT) { const int r = fast_div(e, magC), j = e - r * C; dst[(size_t)(row0 + lr0 + r) * C + j] = zrow[r * pC + j]; }
      }
      if (!last) {
        csync();
        if (tid == 0) st_release_gpu_t(my_flag, it + 1);  // release at gpu scope, cumulative over the CTA barrier above
      }
      TSTAMP(8);
    }
    cluster.sync();  // the peer may still be reading this CTA's partial sums / writing state of the tile's last frame
  }
  if (timing)
    printf("core_fwd_pipe_tc stage %d: frames %d cycles/frame: flagchk %lld | wait_x+actnorm %lld | invconv %lld | z1+syncA %lld | mma_z wait %lld | gate math %lld | sync %lld | LZ+syncB %lld | coupling+publish %lld\n",
           stage, it, tacc[0] / it, tacc[1] / it, tacc[2] / it, tacc[3] / it, tacc[4] / it, tacc[5] / it, tacc[6] / it, tacc[7] / it, tacc[8] / it);
  fence_before();
  __syncthreads();
  if (mma_warp) {
    fence_after();
    tmem_dealloc(tmem, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------
bool pipe_tc_supported(const Dims &d) { return plan_tc(d).total <= 227 * 1024; }

int launch_fwd_pipe_tc(const FwdArgs &a, cudaStream_t st) {
  LFI_REQUIRE(a.stash_tiled, LFI_ERR_ARG, "tensor-core forward pipeline needs the tiled stash");
  static const int timing = getenv("LFI_CORE_TIMING") ? atoi(getenv("LFI_CORE_TIMING")) : 0;
  if (timing) cudaMemcpyToSymbolAsync(g_core_timing, &timing, sizeof(int), 0, cudaMemcpyHostToDevice, st);
  const int nk = a.k_last - a.k_first + 1;
  if (a.h0 || a.h_last) {
    LFI_REQUIRE(a.h0 && a.h_last, LFI_ERR_ARG, "core_fwd_pipe_tc: a carried state needs both h0 and h_last");
    return launch_pipe(core_fwd_pipe_tc<true>, a, FNT, plan_tc(a.d).total, nk, nk, "core_fwd_pipe_tc", st);
  }
  return launch_pipe(core_fwd_pipe_tc<false>, a, FNT, plan_tc(a.d).total, nk, nk, "core_fwd_pipe_tc", st);
}

}  // namespace core
}  // namespace lfi
