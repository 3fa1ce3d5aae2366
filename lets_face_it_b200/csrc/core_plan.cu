// Which flow-core kernels run.  Whole-sequence training picks one kernel per direction here (plan_core), time-chunked evaluation
// its forward kernel (plan_core_eval), the sampler its inverse kernel (use_inv_rows); the launchers run what they are given.
// The switches of DESIGN.md §9 that select these paths are read here only, at call time (the tests toggle them between calls).
#include "core_pipe.cuh"

namespace lfi {
namespace core {

int sm_count() {
  constexpr int kMaxDev = 64;
  static int n[kMaxDev] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= kMaxDev) dev = 0;
  if (n[dev] <= 0) {
    cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev);
    if (n[dev] <= 0) n[dev] = 148;  // no device to ask (workspace sizing on a host without one): a B200's count
  }
  return n[dev];
}

// fwd                                                  bwd
//   PipeTc      tiled                                    PipeTc      tiled, the tensor-core backward fits, LFI_CORE_TC_BWD
//   Pipe        the forward pipeline fits                Pipe        the backward pipeline fits
//   WaveHybrid  tensor-core mode, no forward pipeline,   WaveHybrid  as the forward
//               H % 8 == 0, GH % 16 == 0, B >= 16, LFI_WAVE_TC
//   Wave        otherwise                                Wave        otherwise
// LFI_CORE_PIPE=0 counts as "does not fit" for both pipelines; tiled needs planes and the tensor-core forward (LFI_CORE_TC).
CorePlan plan_core(const Dims &d, int B, int gemm_mode) {
  const bool pipe = env_flag("LFI_CORE_PIPE", true);
  const bool pipe_fwd = pipe && pipe_supported(d, false), pipe_bwd = pipe && pipe_supported(d, true);
  const bool tc = gemm_mode != LFI_GEMM_FP32;
  CorePlan p;
  p.planes = tc && pipe_fwd && pipe_bwd && d.C % 8 == 0 && d.Co % 8 == 0 && d.H % 8 == 0 && d.D % 8 == 0;
  p.tiled = p.planes && env_flag("LFI_CORE_TC", true) && pipe_tc_supported(d);
  const bool hybrid = tc && !pipe_fwd && d.H % 8 == 0 && d.GH % 16 == 0 && B >= 16 && env_flag("LFI_WAVE_TC", true);
  const CoreKernel wave = hybrid ? CoreKernel::WaveHybrid : CoreKernel::Wave;
  p.fwd = p.tiled ? CoreKernel::PipeTc : pipe_fwd ? CoreKernel::Pipe : wave;
  const bool bwd_tc = p.tiled && env_flag("LFI_CORE_TC_BWD", true) && pipe_bwd_tc_supported(d);
  p.bwd = bwd_tc ? CoreKernel::PipeTc : pipe_bwd ? CoreKernel::Pipe : wave;
  return p;
}

// Time-chunked evaluation (lfi_seq_eval): the forward kernel and operand-plane choice of training, run from a carried state.  The
// hybrid wavefronts take no initial state, so their shapes run the plain wavefronts.  (No backward pass: bwd repeats fwd.)
CorePlan plan_core_eval(const Dims &d, int B, int gemm_mode) {
  CorePlan p = plan_core(d, B, gemm_mode);
  if (p.fwd == CoreKernel::WaveHybrid) p.fwd = CoreKernel::Wave;
  p.bwd = p.fwd;
  return p;
}

bool use_inv_rows(const InvArgs &a) { return env_flag("LFI_INV_ROWS", true) && inv_rows_supported(a); }

}  // namespace core
}  // namespace lfi
