// Implicit-GEMM convolution on tcgen05 tensor cores (sm_100a): what the CTA-pair kernel (conv_tc_pair.cuh), the
// streaming 3x3 kernel (conv_tc_halo2.cuh) and the UMMA probe (umma_probe.cuh) share.
//
// Replaces  tf.nn.conv2d(SAME, stride 1, NHWC, HWIO) + bias + PReLU  of the reference
// (helper/tf_graph.py:104-153 conv2d / build_conv; :238-249 build_pixel_shuffler_layer).
//
// GEMM view:  D[M = 128 pixels (TH x TW patch) per CTA, N = cout (padded to 16)]
//             = sum over taps (ky,kx) and 64-channel chunks of  A_tap[128 x 64] * W_tap[64 x N]
//   * A tiles are fetched by TMA (4-D tiled tensor map over the NHWC fp16 plane, SWIZZLE_128B); TMA zero-fills
//     out-of-image pixels, which IS TF's SAME padding - no bounds handling in the kernels.
//   * fp32-equivalent precision from fp16 tensor cores:  a = a_hi + a_lo,  w*2^s = w_hi + w_lo
//     (each 11-bit significands), D += a_hi*w_hi + a_lo*w_hi + a_hi*w_lo   (3 x kind::f16 UMMA,
//     fp32 accumulation in TMEM).  NPLANES == 1 is the single-pass fp16 "fast" mode.
//   * The tensor core's fp32 accumulator update truncates (round-toward-zero) on every UMMA, a bias that grows
//     linearly with the number of accumulation steps (measured: ~0.5 ulp per UMMA, 3e-3 absolute after the
//     333 UMMAs of CNN2).  K is therefore cut into short segments (`seg_chunks` pipeline stages): each segment
//     accumulates in TMEM from zero, and the epilogue warps add the segment sums into fp32 registers with
//     round-to-nearest ("promotion"), double-buffered against the next segment's UMMAs.
//   * Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer (+TMEM alloc), warps 4..11 = epilogue (registers re-balanced with setmaxnreg)
//     (TMEM -> registers, running fp32 sums, then bias/PReLU/split -> global), persistent CTAs striding
//     over (pixel-tile, column-tile) work items.
#pragma once
#include "common.h"
#include "epilogue.cuh"
#include "ptx.cuh"

namespace dcscn {

constexpr int kEpiWarps = 8;                       // two warps per TMEM lane quadrant, each owning half of the columns
constexpr int kEpiWarp0 = 4;                       // warpgroup 0 = {TMA, MMA, 2 idle}; warpgroups 1.. = epilogue
constexpr int kTcThreads = (kEpiWarp0 + kEpiWarps) * 32;
constexpr int kRegsIssue = 40, kRegsEpilogue = 232;  // setmaxnreg budgets (128*56 + 256*224 <= 64K)
constexpr int kMaxStages = 12;
constexpr int kRdotSmemBytes = 9 * 128 * 4;         // fused R-CNN1 filter taps (d2s_cout <= 128) staged in shared memory
constexpr int kAccStages = 2;
constexpr int kAccStride = 256;  // TMEM columns per accumulator stage
constexpr int kColSplit = kEpiWarps / 4;           // column groups
constexpr int kMaxColChunks = 16 / kColSplit;      // 16-column chunks one epilogue thread accumulates (256 columns total)

template <int KC>
struct TcSmem {
  static constexpr int kRowBytes = KC * 2;                  // 128 (SWIZZLE_128B) or 64 (SWIZZLE_64B)
  static constexpr int kABytes = kTileM * kRowBytes;        // one A plane tile
  static constexpr int kSbo = 8 * kRowBytes;                // 8-row core-matrix group stride
  static constexpr uint64_t kLayout = (KC == 64) ? 2ull : 4ull;  // UMMA LayoutType: SW128 = 2, SW64 = 4
};

// Shared-memory matrix descriptor for a K-major swizzled operand tile (cute::UMMA::SmemDescriptor), split for the issue
// loops: the upper word is constant (SBO [32,46), descriptor version bit 46, swizzle mode [61,64)), the lower word is
// (start address >> 4) | LBO (unused for swizzled K-major).
template <int KC>
__device__ __forceinline__ uint32_t desc_lo_t(uint32_t saddr) {
  return ((saddr & 0x3FFFFu) >> 4) | (1u << 16);
}
template <int KC>
__device__ __forceinline__ uint64_t make_desc64_t(uint32_t lo) {
  constexpr uint32_t hi = (uint32_t)(TcSmem<KC>::kSbo >> 4) | (1u << 14) | ((uint32_t)TcSmem<KC>::kLayout << 29);
  return ((uint64_t)hi << 32) | (uint64_t)lo;
}

// kind::f16 instruction descriptor: fp16 x fp16 -> fp32, A and B K-major, M = 128, N = n_pad.
__device__ __forceinline__ uint32_t make_idesc_f16(int n_pad) {
  return (1u << 4) | ((uint32_t)(n_pad >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
}

}  // namespace dcscn
