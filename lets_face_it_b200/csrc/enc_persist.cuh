// Persistent windowed encoder GRU, forward (ModalityEncoder `enc: rnn`, reference models.py:21-27, 55-69): ALL window steps of a
// tile of 128 windows in ONE launch, the recurrent state resident on chip between the steps (enc_persist.cu).
//
// Row-interleaved ("tiled") layout.  The kernel reads its accumulators out of TMEM with thread = window (TMEM lane), so the
// input projections it reads are stored so that the 32 windows of a warp are contiguous per 4-float (16-byte) column group -
// a warp-wide 128-bit access then covers 512 contiguous bytes instead of 32 separate lines:
//   fp32, width W (W % 4 == 0):  element (m, n) at ((m >> 5) * (W >> 2) + (n >> 2)) * 128 + (m & 31) * 4 + (n & 3)       [floats]
// Rows are padded to a multiple of 32.  The input projections xp are TIME-major and tiled (row r = tau * B + b, written
// by the projection GEMM's row-interleaved epilogue, GemmArgs::c_tiled32): the raw frame of window m at step s is then row
// m + (t0 - hist + 1 + s) * B - a constant offset per step, so the 32 windows of a warp read 32 consecutive rows.
#pragma once
#include "lfi_common.cuh"

namespace lfi {
namespace encp {

__host__ __device__ inline size_t tiled_rows(size_t M) { return (M + 31) & ~(size_t)31; }

struct FwdArgs {
  int E, hist, B, T, t0, M;       // hidden size, window length, batch geometry (row m = t' * B + b), rows
  int nplanes;                    // 2 = split-bf16 (three products), 1 = bf16
  const float *xp;                // time-major, tiled [round_up(T*B, 32)][3E]: x @ W_ih^T (no bias), once per raw frame
  const float *b_ih, *b_hh;       // [3E]
  const float *mask;              // [M][hist] frame-dropout mask (already scaled) or nullptr
  const void *whh_hi, *whh_lo;    // bf16 planes of W_hh [3E][E]
  float *cond; int cond_ld;       // final state -> cond[m * cond_ld + e]  (row-major)
  int timing;                     // debug (LFI_ENC_TIMING=1): block (0,0) prints its per-step phase cycles
};

bool fwd_supported(int E, int hist, size_t M, int mode);
int launch_fwd(const FwdArgs &a, cudaStream_t st);

}  // namespace encp

namespace tc {
// gemm_tc.cu: TMA descriptor of a bf16 plane [batch][rows][ldp], box = 64 columns x box_rows rows, 128-byte swizzle
int make_plane_map(void *map, const void *plane, int rows, int cols, int ldp, long stride, int batch, int box_rows);
}  // namespace tc
}  // namespace lfi
