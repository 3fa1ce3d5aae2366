// tcgen05 / TMEM / TMA GEMM for the time-parallel contractions of the conditional-Glow path
// (cond_transform, gate-ih, the windowed encoder GRUs and every weight gradient; reference call sites
// models.py:63-64, 187-190, 206-208 and their autograd).
//
//   C[b] = op(A[b]) op(B[b])  (+ bias, LeakyReLU, LeakyReLU', accumulate)       fp32 in / fp32 out
//
// Numerics (lfi_gemm_mode):
//   BF16   : operands rounded to bf16, one tcgen05.mma.kind::f16 product, fp32 accumulation in TMEM.
//   BF16X3 : operands split a = a_hi + a_lo (two bf16 planes, 16 mantissa bits), three products
//            a_hi b_hi + a_hi b_lo + a_lo b_hi accumulated in the same TMEM tile: fp32-grade
//            (measured 1.4e-6 on z after 16 steps x 56 frames, SURVEY.md §7).
//
// Structure: a persistent, warp-specialised kernel, one CTA per SM.
//   warp 0   : TMA producer   - cp.async.bulk.tensor (128B swizzle) of the A / B planes into a ring of stages
//   warp 1   : MMA issuer     - one thread issues tcgen05.mma (M=128, N=bn<=256, K=16) into one of two TMEM
//                               accumulator tiles and commits stage / accumulator barriers
//   warps 2-9: epilogue       - tcgen05.ld the finished accumulator, transpose through shared memory, fused
//                               epilogue, fully coalesced global stores (or red.add for split-K)
// Large GEMMs run as CTA pairs (2-CTA clusters, tcgen05.mma.cta_group::2): one MMA covers a 256-row tile, each CTA
// stages its 128 rows of A and half of the B tile, the leader CTA issues, completion is committed to both CTAs.
// Both operand majors are native: a row-major [MN, K] plane is a K-major UMMA operand, a row-major [K, MN]
// plane (weight-gradient GEMMs reduce over the rows of two activation matrices) is an MN-major operand, so no
// transposed copies of activations are ever materialised.
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_bf16.h>

#include "lfi_common.cuh"

namespace lfi {
namespace tc {

constexpr int BM = 128;        // tile rows (UMMA M, cta_group::1)
constexpr int BK = 64;         // bf16 elements per k-block = one 128-byte swizzle span
constexpr int UK = 16;         // UMMA K for 16-bit operands
constexpr int kEpiWarps = 12;      // generic epilogue: three warps per TMEM lane quarter take alternate 16-column passes.  12 instead of 8
                                   // (round 2): the epilogue-heavy launches (plane outputs, LeakyReLU', column sums on short K) were bound by
                                   // it - CTA-pair GEMMs of a step 2.13 -> 1.97 ms; 125 registers, no spills; 16 warps would cost a ring stage
constexpr int kGruEpiWarps = 8;   // (16 epilogue warps were measured slower: 96 registers per thread spill, 2.88 vs 2.37 ms per step)
constexpr int kThreads = 64 + 32 * kEpiWarps;  // TMA warp + MMA warp + epilogue warps
__host__ __device__ constexpr int threads_for(int ew) { return 64 + 32 * ew; }
__host__ __device__ constexpr int epi_bytes_for(int ew) { return ew * 32 * 20 * 4; }
constexpr int kMaxStages = 8;
constexpr int kEpiPitch = 20;  // floats; 32 rows x 16 columns per staging pass, conflict-free for 128-bit accesses
constexpr int kTmemCols = 512;  // two accumulator tiles of up to 256 columns
constexpr int kSmemLimit = 225 * 1024;  // dynamic; leaves room for the 1 KB alignment reserve

struct Params {
  int M, N, K, batch;
  int bn;          // tile columns: 64, 128, 192 or 256
  int nplanes;     // 1 = bf16, 2 = split bf16 (three products)
  int a_mn, b_mn;  // 1 = operand stored [K, MN] (MN contiguous)
  int stages, splitk;
  int tiles_m, tiles_n;
  float *C; int ldc; long sC;
  const float *bias; long sBias;
  const float *aux; int ldaux; long sAux;
  int epi;
  // optional bf16 plane output of the final value (hi, and lo = bf16(v - hi) when o_lo != nullptr); C may then be null
  __nv_bfloat16 *o_hi, *o_lo; int ldo; long sO;
  int vec;  // all fp32 pointers / pitches allow 128-bit accesses
  const __nv_bfloat16 *auxp; int ldauxp; long sAuxp;  // LeakyReLU' mask from the sign of a bf16 plane
  float *colsum; long sColsum;                          // += column sums of the final values
  int c_tiled;  // row-interleaved C (GemmArgs::c_tiled32)
  int fuse;     // LFI_FUSE_*
  int cond_vec; // fused GRU forward: the cond slice allows 128-bit stores
  GruEpi gru;
};

// ---- PTX wrappers ------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
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
// Bounded wait: a protocol bug must abort the kernel (sticky error -> LFI_ERR_CUDA), never hang the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  unsigned long long t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  while (!mbar_try_wait(bar, parity)) {
    unsigned long long t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    if (t1 - t0 > 4000000000ull) {
      printf("lfi gemm_tc: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
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

// ---- cta_group::2 (CTA pair) variants -----------------------------------------------------------------
// The two CTAs of a cluster sit on the two SMs of a TPC and execute ONE tcgen05.mma over a 256-row tile: each CTA
// stages its own 128 rows of A and HALF of the B tile, the tensor cores of both SMs read both halves, each CTA's TMEM
// receives its 128 accumulator rows.  Only the leader (cluster rank 0) issues MMAs; TMA loads of both CTAs signal the
// LEADER's full barrier, MMA completion is committed to the barriers of both CTAs.
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void tma_load_3d_2sm(void *smem, const CUtensorMap *map, uint32_t bar_cluster, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem)), "l"((uint64_t)map), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint64_t *bar) {  // arrives on the same barrier in both CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster) : "memory");
}
__device__ __forceinline__ void cluster_arrive_wait() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor (sm_100 UMMA, 128-byte swizzle).  All fields in 16-byte units.
//   K-major  plane tile [rows][64 bf16]: 8-row swizzle atoms of 1024 B  -> SBO = 1024, LBO unused
//   MN-major plane tile: 64-wide MN chunks of [BK rows][64 bf16]        -> SBO = 1024 (8 k-rows), LBO = BK*128
__device__ __forceinline__ uint64_t make_sdesc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= 1ull << 46;  // descriptor version (Blackwell)
  d |= 2ull << 61;  // SWIZZLE_128B
  return d;
}

struct TileCoord { int b, m0, n0, kb0, kb1; };

// CL = 2: the two CTAs of a pair take the row tiles 2i and 2i+1 of the same column tile (a 256-row UMMA tile); with an odd
// number of row tiles the last pair's second half lies outside the matrix (TMA zero fill, epilogue row guard)
__device__ __forceinline__ TileCoord tile_coord(const Params &p, int tile, int nkb, int CL = 1, int rank = 0) {
  // n fastest, then m, then split-k, then batch: CTAs running side by side share the A rows through L2
  TileCoord t;
  const int tn = tile % p.tiles_n; tile /= p.tiles_n;
  const int tmm = (p.tiles_m + CL - 1) / CL;
  const int tm = (tile % tmm) * CL + rank; tile /= tmm;
  const int sk = tile % p.splitk;  tile /= p.splitk;
  t.b = tile; t.m0 = tm * BM; t.n0 = tn * p.bn;
  const int per = (nkb + p.splitk - 1) / p.splitk;
  t.kb0 = sk * per; t.kb1 = min(nkb, t.kb0 + per);
  return t;
}


// ---- fused encoder-GRU epilogues ---------------------------------------------------------------------
__device__ __forceinline__ float4 ld4(const float *p) { return *reinterpret_cast<const float4 *>(p); }
// L2 residency control for the fused encoder-GRU epilogue: the input projections xp (63 MB, re-read by every window step)
// are kept (evict_last) while the write-once stash streams through (evict_first)
__device__ __forceinline__ uint64_t l2_policy_keep() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint64_t l2_policy_stream() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ float4 ld4_hint(const float *p, uint64_t pol) {
  float4 v;
  asm volatile("ld.global.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ void st4_hint(float *p, float a, float b, float c, float d, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d), "l"(pol) : "memory");
}
__device__ __forceinline__ void st2u_hint(void *p, uint2 v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v2.u32 [%0], {%1, %2}, %3;" ::"l"(p), "r"(v.x), "r"(v.y), "l"(pol) : "memory");
}
__device__ __forceinline__ void st4(float *p, float a, float b, float c, float d) { *reinterpret_cast<float4 *>(p) = make_float4(a, b, c, d); }
__device__ __forceinline__ void st_planes4(__nv_bfloat16 *hi, __nv_bfloat16 *lo, size_t o, const float (&v)[4]) {
  __align__(8) __nv_bfloat16 h4[4], l4[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    h4[e] = __float2bfloat16_rn(v[e]);
    l4[e] = __float2bfloat16_rn(v[e] - __bfloat162float(h4[e]));
  }
  *reinterpret_cast<uint2 *>(hi + o) = *reinterpret_cast<const uint2 *>(h4);
  if (lo) *reinterpret_cast<uint2 *>(lo + o) = *reinterpret_cast<const uint2 *>(l4);
}

// One 16-column accumulator chunk: TMEM (thread = row) -> shared-memory transpose -> registers in the "coalesced"
// arrangement of the generic epilogue: lane holds rows rr + 8i (i < 4) x columns cg .. cg+3, so that four lanes cover
// 64 contiguous bytes of a row in every global access.
__device__ __forceinline__ void chunk_to_rows(uint32_t taddr, float *stg, int lane, int rr, int cg, float (&x)[4][4]) {
  uint32_t v[16];
  tmem_ld16(taddr, v);
  tmem_ld_wait();
#pragma unroll
  for (int j = 0; j < 4; ++j)
    *reinterpret_cast<float4 *>(&stg[lane * kEpiPitch + 4 * j]) =
        make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
  __syncwarp();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 t = *reinterpret_cast<const float4 *>(&stg[(rr + 8 * i) * kEpiPitch + cg]);
    x[i][0] = t.x; x[i][1] = t.y; x[i][2] = t.z; x[i][3] = t.w;
  }
  __syncwarp();
}

// Forward (aux::enc_gate_fwd_kernel semantics): tile = 128 windows x 64 hidden units; TMEM columns [0,64) hold the r
// pre-activations of those units, [64,128) u, [128,192) n (the B tile is gathered from the three gate blocks of W_hh).
// Per 16-unit chunk: all global operands are requested first (they do not depend on the accumulator), then the
// accumulator chunks are pulled out of TMEM, then gate math and stores.
template <bool XF>  // XF: the input projections arrive in the accumulator (LFI_FUSE_GRU_FWD_X), columns [3UT,4UT) = n gate's input part
__device__ __forceinline__ void gru_fwd_tile(const Params &p, const TileCoord &t, uint32_t tbase, float *stg, int q, int half, int lane,
                                             uint64_t *tfull, uint32_t aph, int nsub) {
  const GruEpi &G = p.gru;
  const int E = G.E;
  const int rr = lane & 7, cg = (lane >> 3) * 4;
  const int UT = p.bn / 3;  // hidden units per tile (64): TMEM columns [0,UT) r, [UT,2UT) u, [2UT,3UT) n
  const int u_base = (t.n0 / p.bn) * UT;
  const int mrow0 = t.m0 + q * 32;
  __nv_bfloat16 *hhi = (__nv_bfloat16 *)G.h_hi, *hlo = (__nv_bfloat16 *)G.h_lo;
  const uint64_t pol_keep = l2_policy_keep(), pol_stream = l2_policy_stream();
  bool waited = false;
  for (int sc = half; sc < UT / 16; sc += nsub) {
    const int e = min(u_base + 16 * sc + cg, E - 4);
    float4 xr[4], xu[4], xn[4], hp[4];
    float mk[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = min(mrow0 + rr + 8 * i, p.M - 1);
      const int b = m % G.B, tp = m / G.B;
      const int tau = G.t0 + tp - G.hist + 1 + G.s;
      if constexpr (!XF) {
        mk[i] = G.mask ? G.mask[(size_t)m * G.hist + G.s] : 1.0f;
        const float *xp = G.xp + ((size_t)b * G.T + tau) * 3 * E + e;
        xr[i] = ld4_hint(xp, pol_keep); xu[i] = ld4_hint(xp + E, pol_keep); xn[i] = ld4_hint(xp + 2 * E, pol_keep);
      } else {
        mk[i] = 1.0f; xr[i] = xu[i] = make_float4(0.f, 0.f, 0.f, 0.f);  // (already inside the r / u accumulators)
      }
      hp[i] = G.hprev ? ld4(G.hprev + (size_t)m * E + e) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const float4 bir = __ldg(reinterpret_cast<const float4 *>(G.b_ih + e)), biu = __ldg(reinterpret_cast<const float4 *>(G.b_ih + E + e)),
                 bin = __ldg(reinterpret_cast<const float4 *>(G.b_ih + 2 * E + e));
    const float4 bhr = __ldg(reinterpret_cast<const float4 *>(G.b_hh + e)), bhu = __ldg(reinterpret_cast<const float4 *>(G.b_hh + E + e)),
                 bhn = __ldg(reinterpret_cast<const float4 *>(G.b_hh + 2 * E + e));
    if (!waited) { mbar_wait(tfull, aph); tc_fence_after(); waited = true; }
    float ar[4][4], au[4][4], an[4][4];
    chunk_to_rows(tbase + sc * 16, stg, lane, rr, cg, ar);
    chunk_to_rows(tbase + UT + sc * 16, stg, lane, rr, cg, au);
    chunk_to_rows(tbase + 2 * UT + sc * 16, stg, lane, rr, cg, an);
    if constexpr (XF) {
      float ax[4][4];
      chunk_to_rows(tbase + 3 * UT + sc * 16, stg, lane, rr, cg, ax);
#pragma unroll
      for (int i = 0; i < 4; ++i) xn[i] = make_float4(ax[i][0], ax[i][1], ax[i][2], ax[i][3]);
      if (G.x_only) {  // no recurrent product was issued: the h-side n columns of the accumulator were never written
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int c = 0; c < 4; ++c) an[i][c] = 0.f;
      }
    }
    if (u_base + 16 * sc + cg >= E) continue;
    const float bir_[4] = {bir.x, bir.y, bir.z, bir.w}, biu_[4] = {biu.x, biu.y, biu.z, biu.w}, bin_[4] = {bin.x, bin.y, bin.z, bin.w};
    const float bhr_[4] = {bhr.x, bhr.y, bhr.z, bhr.w}, bhu_[4] = {bhu.x, bhu.y, bhu.z, bhu.w}, bhn_[4] = {bhn.x, bhn.y, bhn.z, bhn.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = mrow0 + rr + 8 * i;
      if (m < p.M) {
        const float xr_[4] = {xr[i].x, xr[i].y, xr[i].z, xr[i].w}, xu_[4] = {xu[i].x, xu[i].y, xu[i].z, xu[i].w};
        const float xn_[4] = {xn[i].x, xn[i].y, xn[i].z, xn[i].w}, hp_[4] = {hp[i].x, hp[i].y, hp[i].z, hp[i].w};
        float rg[4], ug[4], ng[4], ah[4], hn[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float air = mk[i] * xr_[c] + bir_[c], aiu = mk[i] * xu_[c] + biu_[c], ain = mk[i] * xn_[c] + bin_[c];
          const float ahr = bhr_[c] + ar[i][c], ahu = bhu_[c] + au[i][c];
          ah[c] = bhn_[c] + an[i][c];
          rg[c] = fast_sigmoid(air + ahr);
          ug[c] = fast_sigmoid(aiu + ahu);
          ng[c] = fast_tanh(ain + rg[c] * ah[c]);
          hn[c] = ng[c] + ug[c] * (hp_[c] - ng[c]);
        }
        const size_t o1 = (size_t)m * E + e, o3 = (size_t)m * 3 * E + e;
        st4(G.h + o1, hn[0], hn[1], hn[2], hn[3]);
        if (G.gates && G.gates16) {
          unsigned short *gq = reinterpret_cast<unsigned short *>(G.gates);
          st2u_hint(gq + o3, make_uint2(q_unorm16(rg[0]) | ((uint32_t)q_unorm16(rg[1]) << 16), q_unorm16(rg[2]) | ((uint32_t)q_unorm16(rg[3]) << 16)), pol_stream);
          st2u_hint(gq + o3 + E, make_uint2(q_unorm16(ug[0]) | ((uint32_t)q_unorm16(ug[1]) << 16), q_unorm16(ug[2]) | ((uint32_t)q_unorm16(ug[3]) << 16)), pol_stream);
          st2u_hint(gq + o3 + 2 * E, make_uint2(q_snorm16(ng[0]) | ((uint32_t)q_snorm16(ng[1]) << 16), q_snorm16(ng[2]) | ((uint32_t)q_snorm16(ng[3]) << 16)), pol_stream);
        } else if (G.gates) {
          st4(G.gates + o3, rg[0], rg[1], rg[2], rg[3]);
          st4(G.gates + o3 + E, ug[0], ug[1], ug[2], ug[3]);
          st4(G.gates + o3 + 2 * E, ng[0], ng[1], ng[2], ng[3]);
        }
        if (G.ahn) st4_hint(G.ahn + o1, ah[0], ah[1], ah[2], ah[3], pol_stream);
        if (G.cond) {
          float *cd = G.cond + (size_t)m * G.cond_ld + e;
          if (p.cond_vec) st4(cd, hn[0], hn[1], hn[2], hn[3]);
          else { cd[0] = hn[0]; cd[1] = hn[1]; cd[2] = hn[2]; cd[3] = hn[3]; }
        }
        if (hhi) st_planes4(hhi, hlo, o1, hn);
      }
    }
  }
  if (!waited) { mbar_wait(tfull, aph); tc_fence_after(); }
}

template <int FUSE, int CL, int EW = kEpiWarps>
__global__ void __launch_bounds__(threads_for(EW), 1)
gemm_tc_kernel(const Params p, const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
               const __grid_constant__ CUtensorMap mapB0, const __grid_constant__ CUtensorMap mapB1,
               const __grid_constant__ CUtensorMap mapXA0, const __grid_constant__ CUtensorMap mapXA1,
               const __grid_constant__ CUtensorMap mapXB0, const __grid_constant__ CUtensorMap mapXB1) {
  constexpr bool GRUF = FUSE == LFI_FUSE_GRU_FWD || FUSE == LFI_FUSE_GRU_FWD_X;   // fused GRU forward (with / without input part)
  constexpr bool XF = FUSE == LFI_FUSE_GRU_FWD_X;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // carve-up: [stages][A planes | B planes] | epilogue staging | barriers | tmem address
  uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const uint32_t a_plane = BM * BK * 2;            // 16 KB
  const uint32_t b_plane = (uint32_t)(p.bn / CL) * BK * 2;  // CTA pair: each CTA stages half of the B tile
  const uint32_t stage_bytes = p.nplanes * (a_plane + b_plane);
  float *epi_stage = (float *)(smem + (size_t)p.stages * stage_bytes);
  uint64_t *bars = (uint64_t *)((uint8_t *)epi_stage + epi_bytes_for(EW));
  uint64_t *full = bars, *empty = bars + kMaxStages, *tfull = bars + 2 * kMaxStages, *tempty = tfull + 2;
  uint32_t *tmem_slot = (uint32_t *)(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb = (p.K + BK - 1) / BK;
  const int ntiles = ((p.tiles_m + CL - 1) / CL) * p.tiles_n * p.splitk * p.batch;  // per cluster
  const int rank = CL > 1 ? (int)cluster_ctarank() : 0;
  const int tile0 = blockIdx.x / CL, tstride = gridDim.x / CL;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < p.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], CL * EW); }  // pair: the leader's collects both epilogues
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  } else if (warp == 1) {
    if constexpr (CL == 2) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (CL > 1) cluster_arrive_wait();  // the peer's barriers are initialised before anything is signalled into them
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      for (int tile = tile0; tile < ntiles; tile += tstride) {
        const TileCoord t = tile_coord(p, tile, nkb, CL, rank);
        const int kb_end = (XF && p.gru.x_only) ? t.kb0 : t.kb1;
        for (int kb = t.kb0; kb < kb_end; ++kb) {
          mbar_wait(&empty[s], ph ^ 1);
          if (CL == 1 || rank == 0) mbar_expect_tx(&full[s], CL * stage_bytes);  // pair: both CTAs' loads land on the leader's barrier
          const uint32_t fbar = CL > 1 ? mapa_u32(smem_u32(&full[s]), 0) : 0;
          uint8_t *sa = smem + (size_t)s * stage_bytes;
          uint8_t *sb = sa + p.nplanes * a_plane;
          const int k0 = kb * BK;
          for (int pl = 0; pl < p.nplanes; ++pl) {
            const CUtensorMap *ma = pl ? &mapA1 : &mapA0;
            const CUtensorMap *mb = pl ? &mapB1 : &mapB0;
            if constexpr (CL == 2) {
              if (!p.a_mn) {
                tma_load_3d_2sm(sa + pl * a_plane, ma, fbar, k0, t.m0, t.b);
              } else {
                for (int j = 0; j < BM / 64; ++j) tma_load_3d_2sm(sa + pl * a_plane + j * (BK * 128), ma, fbar, t.m0 + 64 * j, k0, t.b);
              }
            } else if (!p.a_mn) {
              tma_load_3d(sa + pl * a_plane, ma, &full[s], k0, t.m0, t.b);
            } else {
              for (int j = 0; j < BM / 64; ++j) tma_load_3d(sa + pl * a_plane + j * (BK * 128), ma, &full[s], t.m0 + 64 * j, k0, t.b);
            }
            if (GRUF) {
              // 64 hidden units x (r, u, n): three 64-row boxes of W_hh, 8-row swizzle atoms stay contiguous
              const int ut = p.bn / 3, u0 = (t.n0 / p.bn) * ut;  // (ut rows per gate box)
              for (int g = 0; g < 3; ++g) tma_load_3d(sb + pl * b_plane + g * (ut * 128), mb, &full[s], k0, g * p.gru.E + u0, t.b);
            } else if constexpr (CL == 2) {
              // this CTA stages its half of the B tile: columns [n0 + rank * bn/2, + bn/2)
              const int half = p.bn / 2;
              if (!p.b_mn) {
                tma_load_3d_2sm(sb + pl * b_plane, mb, fbar, k0, t.n0 + rank * half, t.b);
              } else {
                for (int j = 0; j < half / 64; ++j) tma_load_3d_2sm(sb + pl * b_plane + j * (BK * 128), mb, fbar, t.n0 + rank * half + 64 * j, k0, t.b);
              }
            } else if (!p.b_mn) {
              tma_load_3d(sb + pl * b_plane, mb, &full[s], k0, t.n0, t.b);
            } else {
              for (int j = 0; j < p.bn / 64; ++j) tma_load_3d(sb + pl * b_plane + j * (BK * 128), mb, &full[s], t.n0 + 64 * j, k0, t.b);
            }
          }
          if (++s == p.stages) { s = 0; ph ^= 1; }
        }
        if constexpr (XF) {  // input part: k-blocks of [masked window inputs | W_ih], same stage geometry
          const int nxb = (p.gru.xk + BK - 1) / BK;
          const int ut = p.bn / 3, u0 = (t.n0 / p.bn) * ut;
          for (int xb = 0; xb < nxb; ++xb) {
            mbar_wait(&empty[s], ph ^ 1);
            mbar_expect_tx(&full[s], stage_bytes);
            uint8_t *sa = smem + (size_t)s * stage_bytes;
            uint8_t *sb = sa + p.nplanes * a_plane;
            for (int pl = 0; pl < p.nplanes; ++pl) {
              tma_load_3d(sa + pl * a_plane, pl ? &mapXA1 : &mapXA0, &full[s], xb * BK, t.m0, 0);
              for (int g = 0; g < 3; ++g) tma_load_3d(sb + pl * b_plane + g * (ut * 128), pl ? &mapXB1 : &mapXB0, &full[s], xb * BK, g * p.gru.E + u0, 0);
            }
            if (++s == p.stages) { s = 0; ph ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0 && rank == 0) {
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)p.a_mn << 15) | ((uint32_t)p.b_mn << 16) |
                             ((uint32_t)(p.bn >> 3) << 17) | ((uint32_t)((CL * BM) >> 4) << 24);
      const uint32_t a_lbo = p.a_mn ? BK * 128 : 0, b_lbo = p.b_mn ? BK * 128 : 0;
      const uint32_t a_adv = p.a_mn ? (UK * 128) >> 4 : (UK * 2) >> 4;  // descriptor address step per UMMA_K
      const uint32_t b_adv = p.b_mn ? (UK * 128) >> 4 : (UK * 2) >> 4;
      int s = 0; uint32_t ph = 0; int it = 0;
      for (int tile = tile0; tile < ntiles; tile += tstride, ++it) {
        const TileCoord t = tile_coord(p, tile, nkb, CL, rank);
        const int as = it & 1; const uint32_t aph = (it >> 1) & 1;
        mbar_wait(&tempty[as], aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * 256;
        uint32_t acc = 0;
        const int kb_end = (XF && p.gru.x_only) ? t.kb0 : t.kb1;
        for (int kb = t.kb0; kb < kb_end; ++kb) {
          mbar_wait(&full[s], ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + (size_t)s * stage_bytes);
          const uint32_t sb = sa + p.nplanes * a_plane;
          const int nprod = p.nplanes == 2 ? 3 : 1;
          for (int pr = 0; pr < nprod; ++pr) {
            // products: (hi,hi), (hi,lo), (lo,hi)
            const int pa = (pr == 2) ? 1 : 0, pb = (pr == 1) ? 1 : 0;
            const uint64_t ad = make_sdesc(sa + pa * a_plane, a_lbo, 1024);
            const uint64_t bd = make_sdesc(sb + pb * b_plane, b_lbo, 1024);
#pragma unroll
            for (int k = 0; k < BK / UK; ++k) {
              if constexpr (CL == 2) umma_bf16_2sm(d_tmem, ad + (uint64_t)(k * a_adv), bd + (uint64_t)(k * b_adv), idesc, acc);
              else umma_bf16(d_tmem, ad + (uint64_t)(k * a_adv), bd + (uint64_t)(k * b_adv), idesc, acc);
              acc = 1;
            }
          }
          if constexpr (CL == 2) umma_commit_2sm(&empty[s]);  // frees the stage in both CTAs once the MMAs above have read it
          else umma_commit(&empty[s]);
          if (++s == p.stages) { s = 0; ph ^= 1; }
        }
        if constexpr (XF) {
          // input part: r, u columns [0, 2 ut) accumulate on top of the recurrent product; the n gate's input part goes to its own
          // column group [3 ut, 4 ut) (fresh accumulator per tile)
          const int ut = p.bn / 3, nxb = (p.gru.xk + BK - 1) / BK;
          const uint32_t idesc_ru = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)((2 * ut) >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
          const uint32_t idesc_n = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(ut >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
          uint32_t accn = 0;
          for (int xb = 0; xb < nxb; ++xb) {
            mbar_wait(&full[s], ph);
            tc_fence_after();
            const uint32_t sa = smem_u32(smem + (size_t)s * stage_bytes);
            const uint32_t sb = sa + p.nplanes * a_plane;
            const int kleft = p.gru.xk - xb * BK;
            const int nk = kleft >= BK ? BK / UK : (kleft + UK - 1) / UK;  // (the zero-filled tail of the k-block is skipped)
            const int nprod = p.nplanes == 2 ? 3 : 1;
            for (int pr = 0; pr < nprod; ++pr) {
              const int pa = (pr == 2) ? 1 : 0, pb = (pr == 1) ? 1 : 0;
              const uint64_t ad = make_sdesc(sa + pa * a_plane, 0, 1024);
              const uint64_t bd = make_sdesc(sb + pb * b_plane, 0, 1024);
              const uint64_t bdn = make_sdesc(sb + pb * b_plane + 2 * ut * 128, 0, 1024);
              for (int k = 0; k < nk; ++k) {
                umma_bf16(d_tmem, ad + (uint64_t)(k * ((UK * 2) >> 4)), bd + (uint64_t)(k * ((UK * 2) >> 4)), idesc_ru, acc);
                acc = 1;
                umma_bf16(d_tmem + 3 * ut, ad + (uint64_t)(k * ((UK * 2) >> 4)), bdn + (uint64_t)(k * ((UK * 2) >> 4)), idesc_n, accn);
                accn = 1;
              }
            }
            umma_commit(&empty[s]);
            if (++s == p.stages) { s = 0; ph ^= 1; }
          }
        }
        if constexpr (CL == 2) umma_commit_2sm(&tfull[as]);  // accumulator complete (in both CTAs' TMEM)
        else umma_commit(&tfull[as]);
      }
    }
  } else {
    // ===================== epilogue (warps 2 .. 2+EW-1) =====================
    // Warp w may read TMEM lanes [32*(w%4), +32).  EW/4 warps share a lane quarter and take alternate 16-column
    // passes: tcgen05.ld (thread = row) -> shared-memory transpose -> 128-bit global accesses in which four lanes
    // cover 64 contiguous bytes of a row.  Operands of the read-modify-write epilogues are prefetched before the
    // TMEM load so their latency overlaps it.
    const int q = warp & 3, half = (warp - 2) >> 2;
    float *stg = epi_stage + (warp - 2) * 32 * kEpiPitch;
    const int rr = lane & 7, cg = (lane >> 3) * 4;
    const bool want_c = p.C != nullptr;
    const bool rmw = (p.epi & LFI_EPI_ACCUM) && p.splitk == 1;
    const bool rmw_pre = (p.epi & LFI_EPI_ACCUM_PRE) != 0;
    int it = 0;
    for (int tile = tile0; tile < ntiles; tile += tstride, ++it) {
      const TileCoord t = tile_coord(p, tile, nkb, CL, rank);
      const int as = it & 1; const uint32_t aph = (it >> 1) & 1;
      float *C = want_c ? p.C + (size_t)t.b * p.sC : nullptr;
      const float *bias = (p.epi & LFI_EPI_BIAS) ? p.bias + (size_t)t.b * p.sBias : nullptr;
      const float *aux = ((p.epi & LFI_EPI_LRELU_BWD) && !p.auxp) ? p.aux + (size_t)t.b * p.sAux : nullptr;
      const __nv_bfloat16 *auxp = ((p.epi & LFI_EPI_LRELU_BWD) && p.auxp) ? p.auxp + (size_t)t.b * p.sAuxp : nullptr;
      float *colsum = p.colsum ? p.colsum + (size_t)t.b * p.sColsum : nullptr;
      __nv_bfloat16 *ohi = p.o_hi ? p.o_hi + (size_t)t.b * p.sO : nullptr;
      __nv_bfloat16 *olo = p.o_lo ? p.o_lo + (size_t)t.b * p.sO : nullptr;
      const bool has_work = t.kb1 > t.kb0;
      const int mrow0 = t.m0 + q * 32;
      bool waited = false;
      if constexpr (GRUF) {
        const uint32_t tb = tmem_base + ((uint32_t)(q * 32) << 16) + as * 256;
        gru_fwd_tile<XF>(p, t, tb, stg, q, half, lane, &tfull[as], aph, EW / 4);
        waited = true;
      }
      for (int sc = half; sc < p.bn / 16 && FUSE == LFI_FUSE_NONE; sc += EW / 4) {
        const int nc0 = t.n0 + sc * 16;
        if (nc0 >= p.N) break;
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + as * 256 + sc * 16;
        if (p.vec) {
          const int n = nc0 + cg;  // N % 4 == 0 in vec mode: a 4-group is entirely inside or outside
          const bool ncol_ok = n < p.N;
          float4 pre[4];
          if (ncol_ok && (rmw || rmw_pre || aux)) {
            const float *src = (rmw || rmw_pre) ? C : aux;
            const int ld = (rmw || rmw_pre) ? p.ldc : p.ldaux;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int m = mrow0 + rr + 8 * i;
              pre[i] = m < p.M ? *reinterpret_cast<const float4 *>(src + (size_t)m * ld + n) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
          } else if (ncol_ok && auxp) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int m = mrow0 + rr + 8 * i;
              uint2 raw = make_uint2(0u, 0u);
              if (m < p.M) raw = *reinterpret_cast<const uint2 *>(auxp + (size_t)m * p.ldauxp + n);
              // bf16 -> fp32 keeps the sign: value bits in the upper half of the word
              pre[i] = make_float4(__uint_as_float(raw.x << 16), __uint_as_float(raw.x & 0xffff0000u), __uint_as_float(raw.y << 16),
                                   __uint_as_float(raw.y & 0xffff0000u));
            }
          }
          float cs[4] = {0.f, 0.f, 0.f, 0.f};
          float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
          if (bias && ncol_ok) bv = *reinterpret_cast<const float4 *>(bias + n);
          if (!waited) { mbar_wait(&tfull[as], aph); tc_fence_after(); waited = true; }
          uint32_t v[16];
          tmem_ld16(taddr, v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 4; ++j)
            *reinterpret_cast<float4 *>(&stg[lane * kEpiPitch + 4 * j]) =
                make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
          __syncwarp();
          if (ncol_ok) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int r = rr + 8 * i, m = mrow0 + r;
              if (m >= p.M) break;
              float4 x4 = *reinterpret_cast<const float4 *>(&stg[r * kEpiPitch + cg]);
              float x[4] = {x4.x, x4.y, x4.z, x4.w};
              const float b4[4] = {bv.x, bv.y, bv.z, bv.w};
              const float a4[4] = {pre[i].x, pre[i].y, pre[i].z, pre[i].w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                float y = has_work ? x[e] : 0.f;
                if (rmw_pre) y += a4[e];
                y += b4[e];
                if (p.epi & LFI_EPI_LRELU) y = y > 0.f ? y : kLeaky * y;
                if (aux || auxp) y *= (a4[e] > 0.f ? 1.f : kLeaky);
                if (rmw) y += a4[e];
                x[e] = y;
                cs[e] += y;
              }
              if (want_c) {
                float *dst = C + (p.c_tiled ? ((size_t)(m >> 5) * (p.ldc >> 2) + (n >> 2)) * 128 + (m & 31) * 4 + (n & 3) : (size_t)m * p.ldc + n);
                if (p.splitk > 1) {
#pragma unroll
                  for (int e = 0; e < 4; ++e) atomicAdd(dst + e, x[e]);
                } else {
                  *reinterpret_cast<float4 *>(dst) = make_float4(x[0], x[1], x[2], x[3]);
                }
              }
              if (ohi) {
                __align__(8) __nv_bfloat16 h4[4], l4[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  h4[e] = __float2bfloat16_rn(x[e]);
                  l4[e] = __float2bfloat16_rn(x[e] - __bfloat162float(h4[e]));
                }
                const size_t o = (size_t)m * p.ldo + n;
                *reinterpret_cast<uint2 *>(ohi + o) = *reinterpret_cast<const uint2 *>(h4);
                if (olo) *reinterpret_cast<uint2 *>(olo + o) = *reinterpret_cast<const uint2 *>(l4);
              }
            }
          }
          if (colsum) {  // rows of this pass: butterfly over the eight row lanes, one atomic per column
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              cs[e] += __shfl_xor_sync(0xffffffffu, cs[e], 1);
              cs[e] += __shfl_xor_sync(0xffffffffu, cs[e], 2);
              cs[e] += __shfl_xor_sync(0xffffffffu, cs[e], 4);
            }
            if (rr == 0 && ncol_ok) {
#pragma unroll
              for (int e = 0; e < 4; ++e) atomicAdd(colsum + n + e, cs[e]);
            }
          }
          __syncwarp();
        } else {
          // generic path (odd pitches / unaligned bases): thread = row, scalar accesses
          if (!waited) { mbar_wait(&tfull[as], aph); tc_fence_after(); waited = true; }
          uint32_t v[16];
          tmem_ld16(taddr, v);
          tmem_ld_wait();
          const int m = mrow0 + lane;
          if (m < p.M) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int n = nc0 + j;
              if (n >= p.N) break;
              float y = has_work ? __uint_as_float(v[j]) : 0.f;
              if (rmw_pre) y += C[(size_t)m * p.ldc + n];
              if (bias) y += bias[n];
              if (p.epi & LFI_EPI_LRELU) y = y > 0.f ? y : kLeaky * y;
              if (aux) y *= (aux[(size_t)m * p.ldaux + n] > 0.f ? 1.f : kLeaky);
              if (auxp) y *= (__bfloat162float(auxp[(size_t)m * p.ldauxp + n]) > 0.f ? 1.f : kLeaky);
              if (colsum) atomicAdd(colsum + n, y);
              if (want_c) {
                float *dst = C + (p.c_tiled ? ((size_t)(m >> 5) * (p.ldc >> 2) + (n >> 2)) * 128 + (m & 31) * 4 + (n & 3) : (size_t)m * p.ldc + n);
                if (p.splitk > 1) atomicAdd(dst, y);
                else if (p.epi & LFI_EPI_ACCUM) *dst += y;
                else *dst = y;
              }
              if (ohi) {
                const __nv_bfloat16 h = __float2bfloat16_rn(y);
                ohi[(size_t)m * p.ldo + n] = h;
                if (olo) olo[(size_t)m * p.ldo + n] = __float2bfloat16_rn(y - __bfloat162float(h));
              }
            }
          }
        }
      }
      if (!waited) { mbar_wait(&tfull[as], aph); tc_fence_after(); }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CL == 1 || rank == 0) mbar_arrive(&tempty[as]);
        else mbar_arrive_cluster(mapa_u32(smem_u32(&tempty[as]), 0));
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (CL > 1) cluster_arrive_wait();  // no CTA leaves while its peer may still read its operands / signal its barriers
  if (warp == 1) {
    tc_fence_after();
    if constexpr (CL == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

// ---- fp32 -> bf16 planes ------------------------------------------------------------------------
// dst planes are [batch][rows][ldp] with ldp = round_up(cols, 8); padding columns are zero.
__global__ void split_planes_kernel(const float *__restrict__ src, int rows, int cols, int ld, long stride, int batch,
                                    __nv_bfloat16 *__restrict__ hi, __nv_bfloat16 *__restrict__ lo, int ldp) {
  const int groups = ldp / 8;
  const size_t total = (size_t)batch * rows * groups;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int gidx = (int)(idx % groups);
    const size_t rb = idx / groups;
    const int r = (int)(rb % rows), b = (int)(rb / rows);
    const float *s = src + (size_t)b * stride + (size_t)r * ld + gidx * 8;
    float v[8];
    const int c0 = gidx * 8;
    if (c0 + 8 <= cols && (((uintptr_t)s) & 15) == 0) {
      const float4 u = *reinterpret_cast<const float4 *>(s), w = *reinterpret_cast<const float4 *>(s + 4);
      v[0] = u.x; v[1] = u.y; v[2] = u.z; v[3] = u.w; v[4] = w.x; v[5] = w.y; v[6] = w.z; v[7] = w.w;
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = (c0 + e < cols) ? s[e] : 0.f;
    }
    __align__(16) __nv_bfloat16 h[8], l[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      h[e] = __float2bfloat16_rn(v[e]);
      l[e] = __float2bfloat16_rn(v[e] - __bfloat162float(h[e]));
    }
    const size_t o = rb * (size_t)ldp + c0;
    *reinterpret_cast<uint4 *>(hi + o) = *reinterpret_cast<const uint4 *>(h);
    if (lo) *reinterpret_cast<uint4 *>(lo + o) = *reinterpret_cast<const uint4 *>(l);
  }
}

// ---- host side ------------------------------------------------------------------------------------
static PFN_cuTensorMapEncodeTiled_v12000 encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (PFN_cuTensorMapEncodeTiled_v12000)p;
  }
  return fn;
}

// plane: bf16 [batch][rows][ldp]; K-major operand: rows = MN extent, cols = K; MN-major: rows = K, cols = MN.
static int make_map(CUtensorMap *map, const __nv_bfloat16 *plane, int rows, int cols, int ldp, long stride, int batch, int box_rows) {
  auto fn = encode_fn();
  LFI_REQUIRE(fn, LFI_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)batch};
  cuuint64_t strides[2] = {(cuuint64_t)ldp * 2, (cuuint64_t)(batch > 1 ? stride : (long)rows * ldp) * 2};
  cuuint32_t box[3] = {64, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, (void *)plane, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  LFI_REQUIRE(r == CUDA_SUCCESS, LFI_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d): rows=%d cols=%d ldp=%d batch=%d box_rows=%d", (int)r, rows,
              cols, ldp, batch, box_rows);
  return LFI_OK;
}

int make_plane_map(void *map, const void *plane, int rows, int cols, int ldp, long stride, int batch, int box_rows) {
  return make_map((CUtensorMap *)map, (const __nv_bfloat16 *)plane, rows, cols, ldp, stride, batch, box_rows);
}

static int choose_bn(int N) {
  int best = 64, waste = round_up(N, 64);
  const int cand[4] = {64, 128, 192, 256};
  for (int i = 0; i < 4; ++i) {
    const int w = round_up(N, cand[i]);
    if (w <= waste) { waste = w; best = cand[i]; }
  }
  return best;
}

struct Operand {
  const __nv_bfloat16 *hi, *lo;
  int rows, cols, ldp;  // plane geometry
  long stride;
  int mn;               // MN-major?
};

static int g_sms = 0;

// Core launch on prepared planes.
static int launch_core(const Operand &A, const Operand &B, const GemmArgs &g, int nplanes, cudaStream_t st) {
  Params p;
  memset(&p, 0, sizeof(p));
  p.M = g.M; p.N = g.N; p.K = g.K; p.batch = g.batch;
  p.bn = choose_bn(g.N);
  p.fuse = g.fuse; p.gru = g.gru;
  const bool gruf = g.fuse == LFI_FUSE_GRU_FWD || g.fuse == LFI_FUSE_GRU_FWD_X;
  if (gruf) {
    LFI_REQUIRE(g.gru.E % 64 == 0 && g.N == 3 * g.gru.E && !B.mn && g.batch == 1, LFI_ERR_SHAPE, "gemm_tc: fused GRU forward needs E %% 64 == 0");
    p.bn = 192;  // 64 hidden units per tile
    if (g.fuse == LFI_FUSE_GRU_FWD_X)
      LFI_REQUIRE(g.gru.xa_hi && g.gru.xb_hi && (nplanes == 1 || (g.gru.xa_lo && g.gru.xb_lo)) && g.gru.xk >= 8 && g.gru.xk % 8 == 0 &&
                      g.gru.xa_ld % 8 == 0 && g.gru.xb_ld % 8 == 0,
                  LFI_ERR_ARG, "gemm_tc: fused GRU forward with input part needs the input / W_ih operand planes (pitch %% 8 == 0)");
    const float *cd = g.gru.cond;
    p.cond_vec = cd && (((uintptr_t)cd & 15) == 0) && g.gru.cond_ld % 4 == 0;
  }
  p.nplanes = nplanes; p.a_mn = A.mn; p.b_mn = B.mn;
  if (!g_sms) {
    int dev = 0;
    LFI_CUDA(cudaGetDevice(&dev));
    LFI_CUDA(cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  // CTA pairs (cta_group::2, 256-row UMMA tiles): each CTA stages half of the B tile, which halves the operand bytes an SM
  // pulls from L2 per MMA cycle - the bound of the 128-row tiles in the split-bf16 mode (64 B/clk/SM needed, ~43 available).
  // Needs a B tile that splits into two halves of whole swizzle atoms (K-major) / 64-wide chunks (MN-major) and enough
  // tiles to fill the machine with pairs.
  bool pair = false;
  if (g.fuse == LFI_FUSE_NONE) {
    int bn2 = p.bn;
    if (B.mn && bn2 % 128 != 0) bn2 = g.N > 128 ? 256 : 128;
    if (!B.mn && bn2 % 16 != 0) bn2 = round_up(bn2, 16);
    const long ptiles = (long)(((g.M + BM - 1) / BM + 1) / 2) * ((g.N + bn2 - 1) / bn2) * g.batch;
    if (g.M > BM && ptiles >= g_sms / 2) { pair = true; p.bn = bn2; }
  }
  if (!pair && g.fuse == LFI_FUSE_NONE && p.bn == 256 && g.N % 128 == 0) {
    // one 128 x 256 tile per CTA and fewer tiles than SMs: the launch is the serial latency of one tile (loads -> MMAs -> epilogue).
    // Half-width tiles give every CTA two or more, so that the mainloop of one overlaps the epilogue of the previous.
    const long t256 = (long)((g.M + BM - 1) / BM) * ((g.N + 255) / 256) * g.batch;
    if (t256 < g_sms && t256 * 2 > g_sms) p.bn = 128;
  }
  const int CL = pair ? 2 : 1;
  p.tiles_m = (g.M + BM - 1) / BM; p.tiles_n = (g.N + p.bn - 1) / p.bn;
  const int stage_bytes = nplanes * (BM * BK * 2 + (p.bn / CL) * BK * 2);  // per CTA
  const int ew = gruf ? kGruEpiWarps : kEpiWarps;
  const int fixed = epi_bytes_for(ew) + (2 * kMaxStages + 4) * 8 + 16 + 1024;
  p.stages = (kSmemLimit - fixed) / stage_bytes;
  if (p.stages > kMaxStages) p.stages = kMaxStages;
  LFI_REQUIRE(p.stages >= 2, LFI_ERR_SHAPE, "gemm_tc: tile does not fit shared memory");
  const int nkb = (g.K + BK - 1) / BK;
  p.splitk = 1;
  const long tiles = (long)((p.tiles_m + CL - 1) / CL) * CL * p.tiles_n * g.batch;  // CTA tiles (pairs: incl. an empty half)
  if (g.epi == LFI_EPI_ACCUM && tiles * 2 <= g_sms && nkb >= 16) {
    int sk = (int)(g_sms / tiles);  // floor: tiles * sk must not spill into a second wave (6 tiles x 25 splits = 150 CTAs did)
    if (sk > nkb / 8) sk = nkb / 8;
    if (sk < 1) sk = 1;
    // every split must own at least one k-block
    const int per = (nkb + sk - 1) / sk;
    sk = (nkb + per - 1) / per;
    p.splitk = sk;
  } else if (g.epi == LFI_EPI_ACCUM && nkb >= 64 && tiles < 4L * g_sms) {
    // a partly filled last wave: pick the split whose tile count quantises best (time ~ waves / split)
    double best = (double)((tiles + g_sms - 1) / g_sms);
    for (int sk = 2; sk <= 8 && sk <= nkb / 16; ++sk) {
      const double cost = (double)((tiles * sk + g_sms - 1) / g_sms) / sk * 1.03;  // small charge for the red.add epilogue
      if (cost < best - 1e-9) { best = cost; p.splitk = sk; }
    }
  }
  p.C = g.C; p.ldc = g.ldc; p.sC = g.sC; p.bias = g.bias; p.sBias = g.sBias; p.aux = g.aux; p.ldaux = g.ldaux; p.sAux = g.sAux;
  p.epi = g.epi;
  p.o_hi = (__nv_bfloat16 *)g.pOut.hi; p.o_lo = (__nv_bfloat16 *)g.pOut.lo; p.ldo = g.pOut.ld; p.sO = g.pOut.stride;
  auto al16 = [](const void *q) { return ((uintptr_t)q & 15) == 0; };
  p.vec = g.N % 4 == 0;
  if (g.C) p.vec = p.vec && al16(g.C) && g.ldc % 4 == 0 && g.sC % 4 == 0;
  if (g.epi & LFI_EPI_BIAS) p.vec = p.vec && al16(g.bias) && g.sBias % 4 == 0;
  p.auxp = (const __nv_bfloat16 *)g.auxp; p.ldauxp = g.ldauxp; p.sAuxp = g.sAuxp; p.colsum = g.colsum; p.sColsum = g.sColsum;
  if ((g.epi & LFI_EPI_LRELU_BWD) && !g.auxp) p.vec = p.vec && al16(g.aux) && g.ldaux % 4 == 0 && g.sAux % 4 == 0;
  if ((g.epi & LFI_EPI_LRELU_BWD) && g.auxp) p.vec = p.vec && (((uintptr_t)g.auxp & 7) == 0) && g.ldauxp % 4 == 0 && g.sAuxp % 4 == 0;
  if (g.colsum) p.vec = p.vec && g.sColsum % 4 == 0;
  p.c_tiled = g.c_tiled32;
  LFI_REQUIRE(!g.c_tiled32 || (!(g.epi & (LFI_EPI_ACCUM | LFI_EPI_ACCUM_PRE)) && g.ldc % 4 == 0 && g.N % 4 == 0), LFI_ERR_ARG,
              "gemm: row-interleaved output needs a plain store epilogue and 4-column groups");
  if (g.pOut.hi) p.vec = p.vec && al16(g.pOut.hi) && (!g.pOut.lo || al16(g.pOut.lo)) && g.pOut.ld % 4 == 0 && g.pOut.stride % 4 == 0;

  CUtensorMap mA0, mA1, mB0, mB1;
  const int a_box = A.mn ? BK : BM, b_box = B.mn ? BK : (gruf ? p.bn / 3 : (pair ? p.bn / 2 : p.bn));
  LFI_TRY(make_map(&mA0, A.hi, A.rows, A.cols, A.ldp, A.stride, g.batch, a_box));
  LFI_TRY(make_map(&mB0, B.hi, B.rows, B.cols, B.ldp, B.stride, g.batch, b_box));
  if (nplanes == 2) {
    LFI_TRY(make_map(&mA1, A.lo, A.rows, A.cols, A.ldp, A.stride, g.batch, a_box));
    LFI_TRY(make_map(&mB1, B.lo, B.rows, B.cols, B.ldp, B.stride, g.batch, b_box));
  } else {
    mA1 = mA0; mB1 = mB0;
  }
  CUtensorMap mXA0 = mA0, mXA1 = mA1, mXB0 = mB0, mXB1 = mB1;  // (placeholders unless the input part is fused)
  if (g.fuse == LFI_FUSE_GRU_FWD_X) {
    const GruEpi &G = g.gru;
    LFI_TRY(make_map(&mXA0, (const __nv_bfloat16 *)G.xa_hi, g.M, G.xk, G.xa_ld, 0, 1, BM));
    LFI_TRY(make_map(&mXB0, (const __nv_bfloat16 *)G.xb_hi, g.N, G.xk, G.xb_ld, 0, 1, p.bn / 3));
    if (nplanes == 2) {
      LFI_TRY(make_map(&mXA1, (const __nv_bfloat16 *)G.xa_lo, g.M, G.xk, G.xa_ld, 0, 1, BM));
      LFI_TRY(make_map(&mXB1, (const __nv_bfloat16 *)G.xb_lo, g.N, G.xk, G.xb_ld, 0, 1, p.bn / 3));
    } else {
      mXA1 = mXA0; mXB1 = mXB0;
    }
  }
  const int smem = p.stages * stage_bytes + fixed;
  static bool attr_set = false;
  if (!attr_set) {
    LFI_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<LFI_FUSE_NONE, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
    LFI_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<LFI_FUSE_NONE, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
    LFI_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<LFI_FUSE_GRU_FWD, 1, kGruEpiWarps>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
    LFI_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<LFI_FUSE_GRU_FWD_X, 1, kGruEpiWarps>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
    attr_set = true;
  }
  const long ntiles = tiles * p.splitk;
  const int grid = (int)(ntiles < g_sms ? ntiles : g_sms);
  // request > half of the SM's shared memory so that two CTAs (each wanting all 512 TMEM columns) never share an SM
  const int smem_req = smem < 120 * 1024 ? 120 * 1024 : smem;
  if (g.fuse == LFI_FUSE_GRU_FWD) gemm_tc_kernel<LFI_FUSE_GRU_FWD, 1, kGruEpiWarps><<<grid, threads_for(kGruEpiWarps), smem_req, st>>>(p, mA0, mA1, mB0, mB1, mXA0, mXA1, mXB0, mXB1);
  else if (g.fuse == LFI_FUSE_GRU_FWD_X) gemm_tc_kernel<LFI_FUSE_GRU_FWD_X, 1, kGruEpiWarps><<<grid, threads_for(kGruEpiWarps), smem_req, st>>>(p, mA0, mA1, mB0, mB1, mXA0, mXA1, mXB0, mXB1);
  else if (pair) {
    // CTA pairs: one 256-row cta_group::2 tile per cluster
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    const long pairs = ntiles / 2;
    int gp = (int)(pairs < g_sms / 2 ? pairs : g_sms / 2);
    cfg.gridDim = dim3(2 * gp, 1, 1); cfg.blockDim = dim3(kThreads, 1, 1); cfg.dynamicSmemBytes = smem_req; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    LFI_CUDA(cudaLaunchKernelEx(&cfg, gemm_tc_kernel<LFI_FUSE_NONE, 2>, p, mA0, mA1, mB0, mB1, mXA0, mXA1, mXB0, mXB1));
  } else gemm_tc_kernel<LFI_FUSE_NONE, 1><<<grid, kThreads, smem_req, st>>>(p, mA0, mA1, mB0, mB1, mXA0, mXA1, mXB0, mXB1);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

static size_t plane_elems(int rows, int cols, int batch) { return round_up_sz((size_t)batch * rows * round_up(cols, 8), 128); }

size_t split_ws_bytes(const GemmArgs &g, int nplanes) {
  const size_t a = g.transA ? plane_elems(g.K, g.M, g.batch) : plane_elems(g.M, g.K, g.batch);
  const size_t b = g.transB ? plane_elems(g.N, g.K, g.batch) : plane_elems(g.K, g.N, g.batch);
  return (a + b) * 2 * nplanes + 1024;
}

static int split(const float *src, int rows, int cols, int ld, long stride, int batch, __nv_bfloat16 *hi, __nv_bfloat16 *lo, cudaStream_t st) {
  const int ldp = round_up(cols, 8);
  const size_t total = (size_t)batch * rows * (ldp / 8);
  const int threads = 256;
  size_t blocks = (total + threads - 1) / threads;
  if (blocks > 148 * 16) blocks = 148 * 16;
  split_planes_kernel<<<(int)blocks, threads, 0, st>>>(src, rows, cols, ld, stride, batch, hi, lo, ldp);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

}  // namespace tc

// fp32 [batch][rows][cols] (pitch ld) -> bf16 planes [batch][rows][round_up(cols, 8)] (hi, and lo when non-null)
int split_to_planes(const float *src, int rows, int cols, int ld, long stride, int batch, void *hi, void *lo, cudaStream_t st) {
  return tc::split(src, rows, cols, ld, stride, batch, (__nv_bfloat16 *)hi, (__nv_bfloat16 *)lo, st);
}

bool gemm_tc_wants(const GemmArgs &g) {
  // tiny contractions stay on the exact fp32 tiles (nothing to win, and the 1x1-conv / LU helpers need fp32)
  // (K = 30, the speech feature width, is fine: the planes are zero padded to a 16-byte pitch and TMA zero-fills the k-block)
  return g.K >= 24 && g.N >= 16 && g.M >= 16 && (double)g.M * g.N * g.K * g.batch >= 2.0e6;
}

int gemm_tc(int mode, const GemmArgs &g, void *ws, size_t ws_bytes, cudaStream_t st, bool *handled) {
  *handled = false;
  if (!g.pA.hi && !g.pB.hi && !gemm_tc_wants(g)) return LFI_OK;  // operands already in plane form always run here
  const int nplanes = mode == LFI_GEMM_BF16X3 ? 2 : 1;
  const size_t need = tc::split_ws_bytes(g, nplanes);
  LFI_REQUIRE((g.pA.hi && g.pB.hi) || (ws && ws_bytes >= need), LFI_ERR_WORKSPACE,
              "gemm_tc: operand-plane workspace too small (%zu < %zu) for %dx%dx%d b=%d", ws_bytes, need, g.M, g.N, g.K, g.batch);
  LFI_REQUIRE((g.A || g.pA.hi) && (g.B || g.pB.hi) && (g.C || g.pOut.hi || g.fuse), LFI_ERR_ARG, "gemm: null operand");
  LFI_REQUIRE(nplanes == 1 || ((!g.pA.hi || g.pA.lo) && (!g.pB.hi || g.pB.lo)), LFI_ERR_ARG, "gemm: split-bf16 mode needs lo planes");
  LFI_REQUIRE(!(g.epi & LFI_EPI_BIAS) || g.bias, LFI_ERR_ARG, "gemm: bias epilogue without bias");
  LFI_REQUIRE(!(g.epi & LFI_EPI_LRELU_BWD) || g.aux || g.auxp, LFI_ERR_ARG, "gemm: lrelu-bwd epilogue without aux");
  // the vector epilogue would fold the old C into the sums when the launch is not split over K, split-K and the scalar
  // epilogue would not: the result would depend on the split count, so the combination is refused
  LFI_REQUIRE(!(g.colsum && (g.epi & LFI_EPI_ACCUM)), LFI_ERR_ARG, "gemm: column sums cannot be combined with the accumulate epilogue");
  // A: transA = 0 -> stored [M, K] (K-major); 1 -> stored [K, M] (MN-major).  B: transB = 1 -> [N, K] (K-major); 0 -> [K, N] (MN-major)
  tc::Operand A, B;
  A.mn = g.transA ? 1 : 0; A.rows = g.transA ? g.K : g.M; A.cols = g.transA ? g.M : g.K;
  B.mn = g.transB ? 0 : 1; B.rows = g.transB ? g.N : g.K; B.cols = g.transB ? g.K : g.N;
  A.ldp = round_up(A.cols, 8); B.ldp = round_up(B.cols, 8);
  A.stride = (long)A.rows * A.ldp; B.stride = (long)B.rows * B.ldp;
  __nv_bfloat16 *base = (__nv_bfloat16 *)(((uintptr_t)ws + 1023) & ~(uintptr_t)1023);
  const size_t ae = tc::plane_elems(A.rows, A.cols, g.batch), be = tc::plane_elems(B.rows, B.cols, g.batch);
  __nv_bfloat16 *a_hi = base, *a_lo = nplanes == 2 ? base + ae : nullptr;
  __nv_bfloat16 *b_hi = base + ae * nplanes, *b_lo = nplanes == 2 ? b_hi + be : nullptr;
  if (g.pA.hi) {
    A.hi = (const __nv_bfloat16 *)g.pA.hi; A.lo = nplanes == 2 ? (const __nv_bfloat16 *)g.pA.lo : nullptr; A.ldp = g.pA.ld; A.stride = g.pA.stride;
  } else {
    LFI_TRY(tc::split(g.A, A.rows, A.cols, g.lda, g.sA, g.batch, a_hi, a_lo, st));
    A.hi = a_hi; A.lo = a_lo;
  }
  if (g.pB.hi) {
    B.hi = (const __nv_bfloat16 *)g.pB.hi; B.lo = nplanes == 2 ? (const __nv_bfloat16 *)g.pB.lo : nullptr; B.ldp = g.pB.ld; B.stride = g.pB.stride;
  } else {
    LFI_TRY(tc::split(g.B, B.rows, B.cols, g.ldb, g.sB, g.batch, b_hi, b_lo, st));
    B.hi = b_hi; B.lo = b_lo;
  }
  LFI_TRY(tc::launch_core(A, B, g, nplanes, st));
  *handled = true;
  return LFI_OK;
}

}  // namespace lfi
