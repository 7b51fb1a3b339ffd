// Shared host/device declarations for the DCSCN sm_100a hot path.
//
// Data layout in HBM (see DESIGN.md "Data layout"):
//   * Activations between tensor-core layers are kept as TWO fp16 planes ("hi" and "lo",
//     value = hi + lo, 22 significand bits) in NHWC order with a padded channel pitch.  Each
//     layer of the feature-extraction stack owns a 16-channel-aligned slot of one shared
//     "concat" buffer, so tf.concat (DCSCN.py:259,281) never materialises.
//   * Weights are pre-packed per layer into the exact shared-memory image a K-major
//     SWIZZLE_128B UMMA operand tile needs (hi and lo fp16 planes, scaled by a power of two).
#pragma once
#include <cstdint>
#include <cuda_fp16.h>

namespace dcscn {

constexpr int kTileM = 128;          // pixels per CTA tile (UMMA M)
constexpr int kMaxSegments = 2;

enum EpilogueMode : int {
  EPI_PLANES = 0,      // fp16 hi/lo planes, same resolution (up to 2 column segments)
  EPI_D2S_F32 = 1,     // depth_to_space scatter into an fp32 NHWC buffer
  EPI_D2S_PLANES = 2,  // depth_to_space scatter into fp16 hi/lo planes
  EPI_D2S_RDOT = 3,    // depth_to_space fused with the per-pixel half of the final cout=1 conv (R-CNN1):
                       // writes, per HR pixel and filter tap, dot(h[pixel, :], w_last[tap, :])
};

struct EpiSegment {
  int col_begin;       // first GEMM column of this segment (multiple of 16)
  int col_end;         // one past the last column written (multiple of 16)
  __half* dst_hi;      // plane base, already offset to the slot's first channel
  __half* dst_lo;      // may be null in single-plane (fast) mode
  int pitch;           // channels per pixel of the destination buffer (elements)
  __half* dst_zneg;    // training only (else null): fp16 plane, same indexing, of min(z, 0) - the pre-activation's negative
                       // part.  PReLU's backward needs sign(z) and, for d alpha, z itself where z < 0; the post-activation
                       // output cannot give either when the slope alpha is <= 0 (trained checkpoints have many such).
};

struct EpiParams {
  const float* bias;   // [n_total_pad]  (zeros where the layer has no bias / padding)
  const float* alpha;  // [n_total_pad]  PReLU slope; 1.0 == linear layer
  float out_scale;     // 1 / weight_scale (exact power of two)
  int mode;
  int n_valid;         // real output channels (cout) - columns >= n_valid are dropped for D2S
  EpiSegment seg[kMaxSegments];
  int num_seg;
  // depth_to_space
  int d2s_r;           // block size
  int d2s_cout;        // channels after depth_to_space
  float* dst_f32;      // EPI_D2S_F32 destination [N, r*H, r*W, d2s_pitch]
  int d2s_pitch;
  // EPI_D2S_RDOT: final conv weights [taps][d2s_cout] and tap-planar output [taps][N][rH][rW]
  const float* rdot_w;
  float* rdot_out;
  int rdot_taps;
  int rdot_parts;      // epilogue threads sharing one sub-pixel's channels each write their own partial plane set
                       // [parts][taps][N][rH][rW] (1 when a thread's column share covers whole sub-pixels)
  // inverted dropout (training): keep-mask generated from a counter hash; keep_prob==1 -> off
  float keep_prob;
  uint32_t drop_seed;
  uint32_t drop_layer;
  int drop_ntotal;     // channel count the keep-mask index is built with (the slot width; 0 = the GEMM's padded N)
  int store_mode;      // fp16 plane stores of the tensor-core epilogues: 0 = one 32-byte store per lane and plane (default),
                       // 1 = two 16-byte stores (rounds 1-2), 2 = 32-byte stores with neighbouring lanes exchanging halves so
                       // that one instruction covers 64 contiguous bytes of a pixel (streaming 3x3 kernel)
};

struct ConvGeom {
  int n_img, H, W;       // input == output resolution of this conv
  int tiles_x, tiles_y;  // ceil(W/TW), ceil(H/TH)
  int TW, TH;            // TW*TH == 128
};

struct ConvTCParams {
  ConvGeom g;
  int ksz;               // 1 or 3
  int cin_pad;           // padded input channels of the source slot (multiple of 16)
  int chunks;            // ceil(cin_pad / 64)
  int n_tiles;           // column tiles (N > 256 is split)
  int n_pad;             // columns per tile, multiple of 16, <= 256
  int seg_chunks;        // pipeline stages per accumulation segment (fp32 promotion period)
  // streaming kernel (conv_tc_halo2.cuh)
  int h2_nstages;        // weight stages of one (pixel tile, column tile) item: 9 per channel chunk
  int h2_nseg;           // fp32-promotion segments per item
  int h2_resident;       // all stages fit in shared memory: loaded once per CTA
  int pair_stream;       // conv_tc_pair_kernel: streaming split-accumulator mode (1x1 layers)
  unsigned long long* dbg;   // diagnostic builds (-DDCSCN_H2_DEBUG): per-cluster wait counters, else null
  EpiParams epi;
};

// Parameters of the CUDA-core validation convolution (same math in plain fp32 FMAs).
struct ConvRefParams {
  ConvGeom g;
  int ksz;
  int cin;               // logical input channels
  int cout;              // logical output channels
  const __half* src_hi;  // input planes, already offset to the slot
  const __half* src_lo;
  int src_pitch;
  const int* in_map;     // [cin] channel position inside the source buffer
  const float* w;        // HWIO fp32 [k][k][cin][cout]
  int n_total_pad;
  EpiParams epi;         // out_scale must be 1 for this path
};

}  // namespace dcscn
