// Persistent windowed encoder GRU, forward only (ModalityEncoder `enc: rnn`: a one-layer batch-first nn.GRU run from a zero state
// over the `history` frames of every window, reference models.py:21-27 and 55-69; gate equations of torch nn.GRU, order r, z, n).
// Sampling and feature encoding use it; training runs the per-step launches, which also write the stash of the backward pass.
//
// The per-step form runs one launch per window step (recurrent product + gate math), so the state h, its operand planes and the
// input projections make a round trip through HBM / L2 once per step.  Here ONE launch per modality walks all window steps:
//   * a 2-CTA thread-block cluster owns a tile of 128 windows (rows m = t' * B + b) for the whole window; CTA c owns the hidden
//     units [c * E/2, (c+1) * E/2), i.e. the r, u, n columns of those units (3 E/2 <= 384 fp32 accumulator columns in TMEM);
//   * the state h lives in shared memory as split-bf16 (hi, lo) operand planes in the canonical K-major 128-byte-swizzled UMMA
//     layout: it is the A operand of the next step's tcgen05.mma and (hi + lo, exact to 2^-17) the h_{s-1} of the state update.
//     Each CTA writes its half of the new state into its own planes and, through distributed shared memory, into its peer's;
//   * W_hh (this CTA's 3 E/2 rows, both planes) streams from L2 through a TMA ring (cp.async.bulk.tensor, 128-byte swizzle) that
//     runs ahead across step boundaries; one elected thread issues the MMAs (a = a_hi + a_lo: a_hi b_hi + a_lo b_hi + a_hi b_lo,
//     fp32 accumulation in TMEM), eight warps do the gate math straight from TMEM (thread = window x 16-unit chunks);
//   * the input projections xp are read from L2 (63 MB for the widest modality, re-used by every window that contains the
//     frame) in the row-interleaved layout of enc_persist.cuh, so that the thread-per-window accesses of a warp are contiguous
//     (row-major: 32 lines per warp access).  Only the final state leaves the kernel, into the cond columns.
// Synchronisation per step: mbarriers only (no cluster-wide barrier): `a_ready` (16 warp arrivals: both CTAs have written
// their halves of h_s into THIS CTA's planes and this CTA's accumulator reads are done) gates the next product; `mma_done`
// (2 arrivals: this CTA's and the peer's products of the step have completed, so nobody reads h_{s-1} any more) gates the
// state writes.  All waits are bounded (trap after 4 s).
#include "enc_persist.cuh"
#include "tc_ptx.cuh"

#include <cooperative_groups.h>
#include <cuda.h>

namespace cg = cooperative_groups;

namespace lfi {
namespace encp {

using namespace tcp;

namespace {

constexpr int kRows = 128;            // windows per cluster tile (UMMA M)
constexpr int kKB = 64;               // bf16 elements per k-block (one 128-byte swizzle span)
constexpr int kAKB = kRows * 128;     // bytes of one k-block of one A plane
constexpr int kTmemCols = 512;
// The gate phase is issue-latency bound (ncu: 2 gate warps per scheduler sustain ~0.3 instructions per cycle), but 16 gate warps
// (4 per scheduler, 96 registers each) measured slower than 8.
constexpr int kFwdGateWarps = 8;
constexpr int kFwdThreads = 32 * (kFwdGateWarps + 2);  // + TMA producer warp + MMA issuer warp

__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// arrive (release, cluster scope) on a barrier of any CTA of the cluster, given its shared::cluster address
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t *bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// bounded wait on a barrier whose arrivals come from both CTAs of the cluster (mbarrier.arrive.release.cluster).  The wait
// itself uses the default (CTA-scope) acquire: the data it guards lives in THIS CTA's shared memory (written by the peer
// through DSMEM before its release-arrive), and a cluster-scope acquire makes the compiler invalidate L1 (CCTL.IVALL) on every
// spin iteration - 21 % of the stall samples of the first version (profiles/r02_enc_persist_ncu.txt).  Same pattern as the
// CTA-pair GEMM (gemm_tc.cu) and CUTLASS' ClusterBarrier::wait.
__device__ __forceinline__ void mbar_wait_cluster(uint64_t *bar, uint32_t parity) {
  if (mbar_try_wait_cluster(bar, parity)) return;
  unsigned long long t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  while (!mbar_try_wait_cluster(bar, parity)) {
    unsigned long long t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    if (t1 - t0 > 4000000000ull) {
      printf("lfi enc_persist: mbarrier wait timed out (block %d,%d thread %d)\n", blockIdx.x, blockIdx.y, threadIdx.x);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_3d(void *smem, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ float bf_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
__device__ __forceinline__ void unpack8(const uint4 &hi, const uint4 &lo, float *v) {  // v[i] = hi[i] + lo[i]
  v[0] = bf_lo(hi.x) + bf_lo(lo.x); v[1] = bf_hi(hi.x) + bf_hi(lo.x);
  v[2] = bf_lo(hi.y) + bf_lo(lo.y); v[3] = bf_hi(hi.y) + bf_hi(lo.y);
  v[4] = bf_lo(hi.z) + bf_lo(lo.z); v[5] = bf_hi(hi.z) + bf_hi(lo.z);
  v[6] = bf_lo(hi.w) + bf_lo(lo.w); v[7] = bf_hi(hi.w) + bf_hi(lo.w);
}

constexpr int kStageBytes = 192 * 128;  // forward ring stage: one 64-unit half (r, u, n rows) of one k-block of one W_hh plane
constexpr int kMaxStages = 8;

struct SmemPlan {
  int a_plane;      // bytes of one A plane (E/64 k-blocks)
  int b_off, stages;
  int bar_off, total;
};
__host__ __device__ inline SmemPlan plan(int E) {
  SmemPlan p;
  p.a_plane = (E / kKB) * kAKB;
  p.b_off = 2 * p.a_plane;
  const int budget = 227 * 1024 - 1024 - 256 - p.b_off;
  p.stages = budget / kStageBytes;
  if (p.stages > kMaxStages) p.stages = kMaxStages;
  p.bar_off = p.b_off + p.stages * kStageBytes;
  p.total = p.bar_off + 256 + 1024;  // barriers + alignment reserve
  return p;
}

// L1 policy: with 225 KB of shared memory per CTA the L1 is a few tens of KB.  The input projections pass it
// without allocating; the bias vectors, which every chunk of every step re-reads, are asked to stay (evict-last).
__device__ __forceinline__ float4 ld_stream4(const float *p) {
  float4 v;
  asm volatile("ld.global.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ float4 ld_keep4(const float *p) {
  float4 v;
  asm volatile("ld.global.nc.L1::evict_last.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
// 8 consecutive columns n0 .. n0+7 of row `row` of a tiled fp32 array of width W (enc_persist.cuh)
__device__ __forceinline__ void ldt8(const float *base, size_t row, int n0, int W, float *v) {
  const float *p = base + ((row >> 5) * (size_t)(W >> 2) + (size_t)(n0 >> 2)) * 128 + (row & 31) * 4;
  const float4 t0 = ld_stream4(p), t1 = ld_stream4(p + 128);
  v[0] = t0.x; v[1] = t0.y; v[2] = t0.z; v[3] = t0.w; v[4] = t1.x; v[5] = t1.y; v[6] = t1.z; v[7] = t1.w;
}
__device__ __forceinline__ void ldg8(const float *p, float *v) {
  const float4 t0 = ld_keep4(p), t1 = ld_keep4(p + 4);
  v[0] = t0.x; v[1] = t0.y; v[2] = t0.z; v[3] = t0.w; v[4] = t1.x; v[5] = t1.y; v[6] = t1.z; v[7] = t1.w;
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {  // lane = TMEM lane (row), 8 consecutive columns
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

}  // namespace

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kFwdThreads, 1)
enc_gru_fwd_persist(const FwdArgs a, const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_lo) {
  extern __shared__ __align__(16) uint8_t smraw[];
  uint8_t *smb = (uint8_t *)(((uintptr_t)smraw + 1023) & ~(uintptr_t)1023);
  cg::cluster_group cluster = cg::this_cluster();
  const int c = (int)cluster.block_rank();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int E = a.E, UH = E >> 1, NH = UH >> 6, nkb = E / kKB, hist = a.hist;
  const SmemPlan pl = plan(E);
  uint8_t *sA = smb, *sB = smb + pl.b_off;
  uint64_t *bars = (uint64_t *)(smb + pl.bar_off);
  uint64_t *full = bars, *empty = bars + kMaxStages, *mma_local = bars + 2 * kMaxStages, *mma_done = mma_local + 1, *a_ready = mma_local + 2;
  uint32_t *tmem_slot = (uint32_t *)(mma_local + 3);
  uint8_t *peerA = cluster.map_shared_rank(smb, c ^ 1);

  if (tid == 0) {
    for (int s = 0; s < pl.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(mma_local, 1);
    mbar_init(mma_done, 2);                // this CTA's relay + the peer's
    mbar_init(a_ready, 2 * kFwdGateWarps);     // every gate warp of both CTAs
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kFwdGateWarps + 1) tmem_alloc(tmem_slot, kTmemCols);
  fence_before();
  __syncthreads();
  cluster.sync();  // both CTAs run and their barriers are initialised before any remote access
  fence_after();
  const uint32_t tmem = *tmem_slot;
  const int tile = blockIdx.y;
  const uint32_t my_rank = (uint32_t)c, peer_rank = (uint32_t)(c ^ 1);

  if (warp == kFwdGateWarps) {
    // ============================== TMA producer: this CTA's rows of W_hh: k-block, plane, 64-unit half ====================
    if (lane == 0) {
      int st = 0; uint32_t ph = 0;
      for (int s = 1; s < hist; ++s)
        for (int kb = 0; kb < nkb; ++kb)
          for (int p = 0; p < a.nplanes; ++p)
            for (int hf = 0; hf < NH; ++hf) {
              mbar_wait(&empty[st], ph ^ 1);
              mbar_expect_tx(&full[st], (uint32_t)kStageBytes);
              uint8_t *dst = sB + (size_t)st * kStageBytes;
              const CUtensorMap *mp = p ? &map_lo : &map_hi;
#pragma unroll
              for (int g = 0; g < 3; ++g) tma_load_3d(dst + g * 64 * 128, mp, &full[st], kb * kKB, g * E + c * UH + hf * 64, 0);
              if (++st == pl.stages) { st = 0; ph ^= 1; }
            }
    }
  } else if (warp == kFwdGateWarps + 1) {
    // ============================== MMA issuer ==============================================================================
    if (lane == 0) {
      const uint32_t sAu = smem_u32(sA), sBu = smem_u32(sB);
      const uint32_t done_own = mapa_u32(smem_u32(mma_done), my_rank), done_peer = mapa_u32(smem_u32(mma_done), peer_rank);
      const uint32_t idesc = idesc_bf16_m128(192);
      int st = 0; uint32_t ph = 0;
      const bool tm = (a.timing & 1) && blockIdx.x == 0 && blockIdx.y == 0;
      long long t_wait = 0, t_mma = 0;
      for (int s = 1; s < hist; ++s) {
        const long long c0 = tm ? clock64() : 0;
        mbar_wait_cluster(a_ready, (uint32_t)((s - 1) & 1));  // h_{s-1} complete in this CTA's planes, accumulators drained
        const long long c1 = tm ? clock64() : 0;
        t_wait += c1 - c0;
        fence_after();
        fence_async_smem();
        for (int kb = 0; kb < nkb; ++kb)
          for (int p = 0; p < a.nplanes; ++p)
            for (int hf = 0; hf < NH; ++hf) {
              mbar_wait(&full[st], ph);
              fence_after();
              const uint32_t bbase = sBu + (uint32_t)st * kStageBytes;
              // plane 0 (b_hi): a_hi b_hi (+ a_lo b_hi in the split mode); plane 1 (b_lo): a_hi b_lo
              const int na = (p == 0 && a.nplanes == 2) ? 2 : 1;
              for (int pa = 0; pa < na; ++pa) {
                const uint32_t abase = sAu + (uint32_t)pa * pl.a_plane + (uint32_t)kb * kAKB;
#pragma unroll
                for (int ks = 0; ks < kKB / 16; ++ks) {
                  const uint32_t acc = (kb > 0 || p > 0 || pa > 0 || ks > 0) ? 1u : 0u;
                  umma_bf16(tmem + hf * 192, make_sdesc(abase + ks * 32, 1024, kSw128), make_sdesc(bbase + ks * 32, 1024, kSw128), idesc, acc);
                }
              }
              umma_commit(&empty[st]);  // the stage is free once the products above have read it
              if (++st == pl.stages) { st = 0; ph ^= 1; }
            }
        umma_commit(mma_local);
        mbar_wait(mma_local, (uint32_t)((s - 1) & 1));  // this CTA's products of step s are complete ...
        mbar_arrive_cluster(done_own);                  // ... tell this CTA's and the peer's gate warps
        mbar_arrive_cluster(done_peer);
        if (tm) t_mma += clock64() - c1;
      }
      if (tm && hist > 1) printf("enc_persist fwd E=%d hist=%d: MMA warp per step: wait a_ready %lld cycles, products %lld cycles\n", E, hist, t_wait / (hist - 1), t_mma / (hist - 1));
    }
  } else {
    // ============================== gate math: thread = window (TMEM lane) x a quarter of the cluster's hidden units ==========
    const int q = warp & 3, sub = warp >> 2;
    const int L = 32 * q + lane;                // row of the tile = TMEM lane
    const size_t m_raw = (size_t)tile * kRows + L;
    const bool row_ok = m_raw < (size_t)a.M;
    const size_t m = row_ok ? m_raw : (size_t)a.M - 1;  // clamped: rows beyond M compute on valid addresses and store nothing
    const int UQ = UH / (kFwdGateWarps / 4), nch = UQ / 8;      // chunks of 8 units: the working set fits the 168-register budget without spills
    const uint32_t tlane = tmem + ((uint32_t)(32 * q) << 16);
    const uint32_t ready_own = mapa_u32(smem_u32(a_ready), my_rank), ready_peer = mapa_u32(smem_u32(a_ready), peer_rank);
    const bool cond_vec = a.cond && (((uintptr_t)a.cond & 15) == 0) && (a.cond_ld % 4 == 0);
    const bool tm = (a.timing & 1) && blockIdx.x == 0 && blockIdx.y == 0 && tid == 0;
    long long t_wait = 0, t_epi = 0;
    const int ug_first = c * UH + sub * UQ;
    for (int s = 0; s < hist; ++s) {
      const long long c0 = tm ? clock64() : 0;
      const float mk = a.mask ? __ldg(a.mask + m * hist + s) : 1.0f;
      const size_t xr_row = m + (size_t)(a.t0 - hist + 1 + s) * a.B;  // raw frame of this window at this step (time-major rows)
      const bool lastStep = (s == hist - 1);
      float xr[8], xu[8], xn[8];
      // operands of the first chunk are requested before the wait for the products
      ldt8(a.xp, xr_row, ug_first, 3 * E, xr); ldt8(a.xp, xr_row, E + ug_first, 3 * E, xu); ldt8(a.xp, xr_row, 2 * E + ug_first, 3 * E, xn);
      if (s > 0) {
        mbar_wait_cluster(mma_done, (uint32_t)((s - 1) & 1));
        fence_after();
      }
      const long long c1 = tm ? clock64() : 0;
      t_wait += c1 - c0;
      for (int j = 0; j < nch; ++j) {
        const int ul = sub * UQ + 8 * j, ug = c * UH + ul;
        float ar[8], au[8], an[8], hp[8];
        const uint32_t o0 = (uint32_t)(ug >> 6) * kAKB + sw128_off(L, (ug & 63) >> 3);  // 16-byte piece of these 8 units in a plane
        float bri[8], brh[8], bui[8], buh[8];  // the r / u biases are requested before the accumulators are read ...
        ldg8(a.b_ih + ug, bri); ldg8(a.b_hh + ug, brh); ldg8(a.b_ih + E + ug, bui); ldg8(a.b_hh + E + ug, buh);
        if (s > 0) {
          const uint32_t tcol = (uint32_t)((ul >> 6) * 192 + (ul & 63));  // accumulator columns: per 64-unit half [r | u | n]
          tmem_ld8(tlane + tcol, ar);
          tmem_ld8(tlane + tcol + 64, au);
          tmem_ld8(tlane + tcol + 128, an);
          const uint4 h0 = *reinterpret_cast<const uint4 *>(sA + o0), l0 = *reinterpret_cast<const uint4 *>(sA + pl.a_plane + o0);
          unpack8(h0, l0, hp);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i) { ar[i] = 0.f; au[i] = 0.f; an[i] = 0.f; hp[i] = 0.f; }
        }
        float hn[8], ng[8];
        {
          float bni[8], bnh[8];                // ... the n biases while r and u are computed
          ldg8(a.b_ih + 2 * E + ug, bni); ldg8(a.b_hh + 2 * E + ug, bnh);
#pragma unroll
          for (int i = 0; i < 8; ++i) ar[i] = fast_sigmoid(mk * xr[i] + bri[i] + (ar[i] + brh[i]));          // r
#pragma unroll
          for (int i = 0; i < 8; ++i) au[i] = fast_sigmoid(mk * xu[i] + bui[i] + (au[i] + buh[i]));          // u (z in torch's naming)
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            an[i] += bnh[i];                                                                                // h-side n pre-activation
            ng[i] = fast_tanh(mk * xn[i] + bni[i] + ar[i] * an[i]);                                         // n
            hn[i] = ng[i] + au[i] * (hp[i] - ng[i]);                                                        // h' = (1 - u) n + u h
          }
        }
        if (j + 1 < nch) {  // the next chunk's input projections travel while this chunk's state is packed and stored
          const int ugn = ug + 8;
          ldt8(a.xp, xr_row, ugn, 3 * E, xr); ldt8(a.xp, xr_row, E + ugn, 3 * E, xu); ldt8(a.xp, xr_row, 2 * E + ugn, 3 * E, xn);
        }
        uint4 hi0, lo0;
        split8(hn, hi0, lo0);
        if (!lastStep) {  // new state into the operand planes of both CTAs (nobody reads h_{s-1} any more: mma_done)
          *reinterpret_cast<uint4 *>(sA + o0) = hi0; *reinterpret_cast<uint4 *>(sA + pl.a_plane + o0) = lo0;
          *reinterpret_cast<uint4 *>(peerA + o0) = hi0; *reinterpret_cast<uint4 *>(peerA + pl.a_plane + o0) = lo0;
        }
        if (row_ok && lastStep && a.cond) {
          float *cd = a.cond + m * a.cond_ld + ug;
          if (cond_vec) {
            *reinterpret_cast<float4 *>(cd) = make_float4(hn[0], hn[1], hn[2], hn[3]);
            *reinterpret_cast<float4 *>(cd + 4) = make_float4(hn[4], hn[5], hn[6], hn[7]);
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) cd[i] = hn[i];
          }
        }
      }
      if (!lastStep) {
        fence_before();      // this warp's accumulator reads are complete before the next products overwrite them
        fence_async_smem();  // the new state is visible to the tensor cores
        __syncwarp();
        if (lane == 0) { mbar_arrive_cluster(ready_own); mbar_arrive_cluster(ready_peer); }
      }
      if (tm) t_epi += clock64() - c1;
    }
    if (tm) printf("enc_persist fwd E=%d hist=%d: gate warp 0 per step: wait products %lld cycles, gate math + stores %lld cycles\n", E, hist, t_wait / hist, t_epi / hist);
  }

  fence_before();
  __syncthreads();
  cluster.sync();  // no CTA leaves while its peer may still write into its planes or signal its barriers
  if (warp == kFwdGateWarps + 1) {
    fence_after();
    tmem_dealloc(tmem, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------
bool fwd_supported(int E, int hist, size_t M, int mode) {
  if (mode == LFI_GEMM_FP32) return false;
  if (!(E == 128 || E == 256) || hist < 1 || M < 128) return false;
  const SmemPlan p = plan(E);
  return p.stages >= 2 && p.total <= 227 * 1024;
}

int launch_fwd(const FwdArgs &a, cudaStream_t st) {
  LFI_REQUIRE(a.E == 128 || a.E == 256, LFI_ERR_SHAPE, "enc_persist: E=%d unsupported", a.E);
  LFI_REQUIRE(a.xp && a.b_ih && a.b_hh && a.whh_hi && (a.nplanes == 1 || a.whh_lo), LFI_ERR_ARG, "enc_persist: null argument");
  auto al16 = [](const void *p) { return p == nullptr || ((uintptr_t)p & 15) == 0; };
  LFI_REQUIRE(al16(a.xp) && al16(a.b_ih) && al16(a.b_hh), LFI_ERR_ARG, "enc_persist: misaligned pointer");
  const SmemPlan p = plan(a.E);
  LFI_REQUIRE(p.stages >= 2 && p.total <= 227 * 1024, LFI_ERR_SHAPE, "enc_persist: shared-memory plan does not fit");
  CUtensorMap mhi, mlo;
  LFI_TRY(tc::make_plane_map(&mhi, a.whh_hi, 3 * a.E, a.E, a.E, 0, 1, 64));
  if (a.nplanes == 2) LFI_TRY(tc::make_plane_map(&mlo, a.whh_lo, 3 * a.E, a.E, a.E, 0, 1, 64));
  else mlo = mhi;
  static const int timing = env_flag("LFI_ENC_TIMING", false) ? 1 : 0;
  FwdArgs at = a;
  at.timing = timing;
  static bool attr_set = false;
  if (!attr_set) {
    LFI_CUDA(cudaFuncSetAttribute(enc_gru_fwd_persist, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  const int ntiles = (a.M + kRows - 1) / kRows;
  // > half of the SM's shared memory: never two CTAs (each wanting all 512 TMEM columns) on one SM
  const int smem = p.total < 120 * 1024 ? 120 * 1024 : p.total;
  dim3 grid(2, ntiles, 1);
  enc_gru_fwd_persist<<<grid, kFwdThreads, smem, st>>>(at, mhi, mlo);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

}  // namespace encp
}  // namespace lfi
