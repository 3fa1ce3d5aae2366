// Persistent, stage-pipelined flow core (training forward / backward) for GRU coupling networks whose per-step
// weights fit the shared memory of a 2-CTA cluster (final_model.yaml: H = 128, C = 56).
//
// One cluster of two CTAs owns ONE flow step k for the whole launch and keeps that step's weights (W_hh, the z1
// columns of W_ih, LinearZeros, the 1x1 conv) and the RNN state h resident in shared memory across all frames
// (reference: FlowStep.normal_flow models.py:311-342, f_seq.forward models.py:204-214 with the state carried on
// the module, models.py:193-194).  The K clusters of a pipeline form a systolic chain over a tile of 64 sequences:
// stage k evaluates frame t as soon as stage k-1 has published its output for frame t (release/acquire counter in
// global memory), so cell (k, t) runs concurrently with (k-1, t+1), (k-2, t+2), ... - the same anti-diagonal
// schedule as the wavefront kernels (core_fwd.cu / core_bwd.cu), without a launch per diagonal and without
// re-streaming the weights.  Inside a cluster the hidden units are split between the two CTAs (each CTA owns 64
// units = 192 gate columns of W_hh); the halves of h and the LinearZeros partial sums are exchanged through
// distributed shared memory.  The recurrent product h . W_hh^T of frame t does not depend on stage k-1, so it is
// evaluated BEFORE the stage waits for its input: only the small products sit on the stage-to-stage critical path.
#pragma once
#include "core_api.cuh"
#include <cstdio>
#include <cuda_bf16.h>

namespace lfi {
namespace core {

constexpr int PNT = 256;  // threads per CTA
constexpr int PR = 64;    // sequences (rows) per cluster tile
constexpr int PRH = 32;   // rows per CTA for the row-wise work (ActNorm, 1x1 conv, coupling)
constexpr int PUC = 64;   // hidden units per CTA
constexpr int PHS = 68;   // row pitch of the act-layout arrays ([reduction index][row]) over the 64 tile rows

struct PipePlan {  // offsets in floats
  int whh, wz, wf, w, vec, h, z1, xs, zrow, o, extra, total;
  int pC, pO;
};

// forward:  whh [H][3][64] = W_hh[g*H + u][i], wz [Ci][3][64] = W_ih[g*H + u][i], wf [64][Cop] = Wf[j][u], w [C][Cp] = W
// (the backward kernel has its own plan, core_pipe_bwd.cu)
__host__ __device__ inline PipePlan plan_pipe(const Dims &d) {
  PipePlan p;
  int o = 0;
  auto take = [&](int n) { int r = o; o += round_up(n, 4); return r; };
  p.pC = odd(d.C);
  p.pO = round_up(d.Co, 4) + 4;
  p.whh = take(d.H * 3 * PUC);
  p.wz = take(d.Ci * 3 * PUC);
  p.wf = take(PUC * d.Cop);
  p.w = take(d.C * d.Cp);
  p.vec = take(2 * d.C + 3 * PUC + 2 * d.Co);
  p.h = take(d.H * PHS);
  p.z1 = take(d.Ci * PHS);
  p.xs = take(PRH * p.pC);
  p.zrow = take(PRH * p.pC);
  p.o = take(2 * PRH * p.pO);
  p.extra = 0;
  p.total = o;
  return p;
}

// e / c for a divisor that is constant over the launch (the channel count, 56): one multiply-high instead of the ~20-instruction
// integer division, inside loops that sit on the per-frame critical path.  magic = ceil(2^32 / c); exact for e * (magic * c - 2^32) < 2^32,
// i.e. for every e below 2^32 / c.
__device__ __forceinline__ unsigned div_magic(int c) { return (unsigned)((0x100000000ull + (unsigned)c - 1) / (unsigned)c); }
__device__ __forceinline__ int fast_div(int e, unsigned magic) { return (int)__umulhi((unsigned)e, magic); }

// fp32 -> split-bf16 operand planes (gemm_tc.cu): hi = bf16(v), lo = bf16(v - hi)
__device__ __forceinline__ void put_plane(void *hi, void *lo, size_t idx, float v) {
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  ((__nv_bfloat16 *)hi)[idx] = h;
  if (lo) ((__nv_bfloat16 *)lo)[idx] = __float2bfloat16_rn(v - __bfloat162float(h));
}
__device__ __forceinline__ void put_plane2(void *hi, void *lo, size_t idx, float v0, float v1) {  // idx even
  const __nv_bfloat162 h = __floats2bfloat162_rn(v0, v1);
  *reinterpret_cast<__nv_bfloat162 *>((__nv_bfloat16 *)hi + idx) = h;
  if (lo) *reinterpret_cast<__nv_bfloat162 *>((__nv_bfloat16 *)lo + idx) = __floats2bfloat162_rn(v0 - __low2float(h), v1 - __high2float(h));
}

// Tiled stash (gates / ahn / h) shared by the tensor-core forward pipeline and the backward pipeline:
//   [cell][tile of 64 sequences][CTA c][group hs of 16 hidden units][array][float4 i of the group][64 sequences][4 floats]
// (narr = 3 arrays r, u, n for the gates, 1 for ahn and h).  A warp of the forward kernel holds 32 consecutive sequences, one
// per lane, so each of its stores covers 512 contiguous bytes.  Element (sequence row, unit 64c + 16hs + 4i + e): + 4*row + e.
__host__ __device__ inline size_t stash_tiled_off(size_t cell, int ntiles, int tile, int c, int hs, int narr, int arr, int i) {
  return (((((cell * ntiles + tile) * 2 + c) * 4 + hs) * narr + arr) * 4 + i) * 256;
}

// Row-interleaved gate-ih pre-activations G (written by the gate-ih GEMM epilogue, GemmArgs::c_tiled32): element (m, n)
__host__ __device__ inline size_t g_tiled_off(size_t m, size_t n, size_t ld) { return ((m >> 5) * (ld >> 2) + (n >> 2)) * 128 + (m & 31) * 4 + (n & 3); }

// Bounded spin on a stage-progress counter (release/acquire chain between the stages of a pipeline): waits until *flag > it.
// The chain assumes that every CTA of the launch is resident at the same time (checked on the host before the launch,
// pipe_check_residency); if that ever fails (another context holding SMs, a protocol bug) the wait traps after 4 s and the
// launch returns an error instead of hanging the GPU - the same policy as the mbarrier waits (tc_ptx.cuh: mbar_wait).
__device__ __forceinline__ void spin_wait_gt(const int *flag, int it) {
  auto ld = [&]() { int v; asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory"); return v; };
  if (ld() > it) return;
  unsigned long long t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  while (ld() <= it) {
    unsigned long long t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    if (t1 - t0 > 4000000000ull) {
      printf("lfi flow core: stage flag wait timed out (block %d,%d,%d thread %d, it %d)\n", blockIdx.x, blockIdx.y, blockIdx.z, threadIdx.x, it);
      __trap();
    }
  }
}

// Host check before a stage-pipeline launch: all `clusters` 2-CTA clusters must be co-resident (the stages spin on each other).
// cudaOccupancyMaxActiveClusters accounts for the kernel's registers / shared memory on the current device.
template <typename Kern>
inline int pipe_check_residency(Kern kern, int threads, int smem_bytes, int clusters, const char *what) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2, (unsigned)clusters, 1);
  cfg.blockDim = dim3((unsigned)threads, 1, 1);
  cfg.dynamicSmemBytes = (size_t)smem_bytes;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) {  // query unavailable: the bounded spins still protect the GPU
    cudaGetLastError();
    return LFI_OK;
  }
  LFI_REQUIRE(n >= clusters, LFI_ERR_SHAPE, "%s: %d co-resident clusters needed, the device can hold %d", what, clusters, n);
  return LFI_OK;
}

int sm_count();  // SMs of the current device (core_plan.cu)

// The part the four stage-pipeline launchers share: P pipelines of nk stage clusters (grid 2 x nk x P), as many as the SMs hold
// and the tiles of 64 sequences need; flag_rows progress counters per pipeline and CTA, zeroed before the launch.
template <typename Args>
int launch_pipe(void (*kern)(Args, int, int, int *), const Args &a, int threads, int smem_bytes, int nk, int flag_rows,
                const char *what, cudaStream_t st) {
  const int ntiles = (a.B + PR - 1) / PR;
  int P = sm_count() / (2 * nk);
  if (P > ntiles) P = ntiles;
  const size_t flag_bytes = (size_t)P * flag_rows * 2 * sizeof(int);
  LFI_REQUIRE(a.flags, LFI_ERR_ARG, "%s: no progress flags", what);
  LFI_REQUIRE(P >= 1 && flag_bytes <= a.flags_bytes, LFI_ERR_WORKSPACE, "flow core pipeline: flag buffer too small");
  LFI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  LFI_CUDA(cudaMemsetAsync(a.flags, 0, flag_bytes, st));
  LFI_TRY(pipe_check_residency(kern, threads, smem_bytes, nk * P, what));
  kern<<<dim3(2, nk, P), threads, smem_bytes, st>>>(a, P, ntiles, a.flags);
  LFI_LAUNCH_CHECK();
  return LFI_OK;
}

// Shape-only fit tests of the stage pipelines for whole-sequence training (K stages); each tests what it adds to the one
// before it: pipe_supported, then pipe_tc_supported (forward) and pipe_bwd_tc_supported (backward).  Called by plan_core only.
bool pipe_supported(const Dims &d, bool bwd);
bool pipe_tc_supported(const Dims &d);
bool pipe_bwd_tc_supported(const Dims &d);
int pipe_bwd_smem_bytes(const Dims &d);
int launch_fwd_pipe(const FwdArgs &a, cudaStream_t st);
int launch_bwd_pipe(const BwdArgs &a, cudaStream_t st);
// tensor-core variants (core_pipe_fwd_tc.cu, core_pipe_bwd_tc.cu): gate products as tcgen05.mma on split-bf16 operands
int launch_fwd_pipe_tc(const FwdArgs &a, cudaStream_t st);
int launch_bwd_pipe_tc(const BwdArgs &a, cudaStream_t st);

}  // namespace core
}  // namespace lfi
