// Streaming halo kernel of the 3x3 layers: CTA-pair tcgen05 convolution (see conv_tc_pair.cuh) whose A operand is read
// once per channel chunk for all nine taps, and whose weight stages are released as soon as their products are issued.
//
// A operand: the pixel patch is 16 rows x 8 columns.  Per 64-channel chunk ONE {64, 10, 18, 1} TMA box (the patch and
// its one-pixel halo, 180 smem rows of 128 B) serves all nine taps.  The smem rows are (hy * 10 + hx); tap (dy, dx)
// starts (dy * 10 + dx) rows into the box, and the 16 eight-row groups of the UMMA A operand are 10 rows (1280 B) apart,
// so operand rows are NOT aligned to the 1024-byte swizzle atom.  This relies on the tensor core applying the 128B-swizzle
// XOR on absolute shared-memory address bits [7,10), like TMA does when writing - measured on B200: correct with the
// descriptor base-offset field left 0, wrong with it set to the operand's offset inside the atom.
//
// B operand: one weight stage = one [n_pad/2 rows x 128 bytes] (x planes) operand tile per CTA = the four 16-channel K
// slices of one tap of one chunk.  Stages are ordered [chunk][dx][dy] (host: pair_image in engine.cu); a last chunk with
// 16, 32 or 48 valid channels (cin_pad % 64) issues only its first 1, 2 or 3 slices.
//
// Accumulation: three kind::f16 products per algorithmic MAC (conv_tc.cuh).  The tensor core truncates its fp32
// accumulate on every UMMA, so the K loop of a tile is cut into fp32-promotion segments, and the two kinds of products go
// to DIFFERENT TMEM accumulators - the order of issue inside a stage does not matter for accuracy and no stage is held
// for a second pass (profiles/r1d_conv_tc_ncu_summary.csv: round 1's two-pass 3x3 kernel, which kept a segment's stages
// resident until its dominant pass, left two of five 22 KB ring slots free for prefetch and ran every layer at
// ~4.5 TB/s of TMA traffic into shared memory, tensor pipe 31-50 % active):
//   * segments s = 0..nseg-1 end at (chunk, dx) boundaries; accumulation "slot" j = 0..nseg receives the correction
//     products (a_lo*w_hi, a_hi*w_lo) of segment j-1 FIRST (while it is still small) and the dominant products of
//     segment j afterwards;  slot j is complete at the end of segment j and the epilogue warps add it into their fp32
//     registers with round-to-nearest ("promotion").  nseg + 1 drains per tile.
//   * slots rotate over the TMEM buffers of n_pad columns: with three, during segment s buffer (s % 3) takes dominant
//     products, ((s + 1) % 3) corrections, ((s + 2) % 3) is being drained.  3 * n_pad <= 512 columns -> n_pad <= 160;
//     wider layers are split into column tiles by the engine (choose_tiling) or run on two buffers (option "wide_tiles").
//   * every stage of the weight ring and every A slot is released by the tcgen05.commit that follows its last UMMA,
//     so the whole ring (up to 32 stages) is prefetch depth.
#pragma once
#include "conv_tc_pair.cuh"

namespace dcscn {

constexpr int kHaloTW = 8, kHaloTH = 16;                          // pixel patch of one CTA
constexpr int kHalo1W = kHaloTW + 2;                              // 10 columns
constexpr int kHalo1Rows = (kHaloTH + 2) * kHalo1W;               // 180 rows
constexpr int kHalo1PlaneBytes = ((kHalo1Rows * 128 + 1023) / 1024) * 1024;  // 23552, keeps planes 1024-aligned

__host__ __device__ inline size_t tc_halo1_a_slot_bytes(int nplanes) { return (size_t)nplanes * kHalo1PlaneBytes; }
__host__ __device__ inline size_t tc_halo_b_stage_bytes(int nplanes, int n_pad) {
  return (size_t)nplanes * (size_t)(n_pad / 2) * 128;
}

constexpr int kH2MaxStages = 32;
constexpr int kH2MaxAcc = 4;
constexpr int kH2BarBytes = 2048;        // mbarriers (4 x 32 + 2 x 4) + TMEM slot, with room to spare: the engine sizes the rings from it

__host__ __device__ inline size_t tc_halo2_misc_bytes() { return 1024 + kH2BarBytes + kRdotSmemBytes; }

// -DDCSCN_H2_DEBUG builds a diagnostic library (scripts/r2_h2_timeline.sh): the issuing thread and one epilogue warp
// count the cycles they spend waiting on each kind of barrier and write them to p.dbg[cluster][8].
#ifdef DCSCN_H2_DEBUG
#define H2_T0() const long long h2_t0_ = clock64()
#define H2_ACC(var) var += clock64() - h2_t0_
#else
#define H2_T0()
#define H2_ACC(var)
#endif

template <int NPLANES>
__global__ void __launch_bounds__(kTcThreads, 1)
conv_tc_halo2_kernel(const __grid_constant__ CUtensorMap tm_hi, const __grid_constant__ CUtensorMap tm_lo,
                     const __grid_constant__ CUtensorMap tm_w, const ConvTCParams p, const int num_a, const int num_b) {
  constexpr int KC = 64;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int AH_BYTES = kHalo1PlaneBytes;            // one plane of the 18 x 10 box
  constexpr int A_SLOT = NPLANES * AH_BYTES;
  const int half_rows = p.n_pad >> 1;                   // weight-tile rows staged by each CTA of the pair
  const int BH_BYTES = half_rows * KC * 2;              // one plane of this CTA's weight half
  const int B_STAGE = NPLANES * BH_BYTES;
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + (size_t)num_a * A_SLOT;
  uint64_t* a_full = reinterpret_cast<uint64_t*>(smem_b + (size_t)num_b * B_STAGE);
  uint64_t* a_empty = a_full + kH2MaxStages;
  uint64_t* b_full = a_empty + kH2MaxStages;
  uint64_t* b_empty = b_full + kH2MaxStages;
  uint64_t* acc_full = b_empty + kH2MaxStages;
  uint64_t* acc_empty = acc_full + kH2MaxAcc;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + kH2MaxAcc);
  float* s_rdot = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(a_full) + kH2BarBytes);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;
  const int acc_stride = p.n_pad;                       // TMEM columns between accumulation buffers
  // TMEM buffers: 4 (n_pad <= 128: the next tile never waits for this tile's drains), 3 (<= 160), or 2 for the wide tiles
  // of option "wide_tiles" (<= 256: the issuer waits for the previous slot's drain at every segment boundary)
  const uint32_t nbuf = (4 * p.n_pad <= 512) ? 4u : ((3 * p.n_pad <= 512) ? 3u : 2u);

  if (threadIdx.x == 0) {
    for (int s = 0; s < num_a; ++s) {
      ptx::mbar_init(&a_full[s], 1);
      ptx::mbar_init(&a_empty[s], 1);
    }
    for (int s = 0; s < num_b; ++s) {
      ptx::mbar_init(&b_full[s], 1);
      ptx::mbar_init(&b_empty[s], 1);
    }
    for (int s = 0; s < kH2MaxAcc; ++s) {
      ptx::mbar_init(&acc_full[s], 1);                     // leader's tcgen05.commit (multicast)
      ptx::mbar_init(&acc_empty[s], 2 * kEpiWarps);        // epilogue warps of both CTAs (used on the leader only)
    }
    ptx::fence_barrier_init();
    ptx::fence_proxy_async();
  }
  if (warp == 1) {
    ptx::tmem_alloc_2sm(tmem_slot, 512);
    ptx::tmem_relinquish_2sm();
  }
  if (p.epi.mode == EPI_D2S_RDOT)
    for (int i = threadIdx.x; i < p.epi.rdot_taps * p.epi.d2s_cout; i += blockDim.x) s_rdot[i] = p.epi.rdot_w[i];
  const int nst = p.h2_nstages;                       // weight stages of one item: 9 per channel chunk
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  ptx::tc_fence_after();
  // All 512 columns are allocated, so the allocation starts at lane 0, column 0.  Using the literal 0 keeps every TMEM
  // address warp-uniform for the compiler (uniform registers feed UTCHMMA directly; a value loaded from shared memory costs a
  // vector->uniform move in front of every UMMA of the single issuing thread).
  if (*tmem_slot != 0u) __trap();
  constexpr uint32_t tmem_base = 0u;
  const bool resident = p.h2_resident != 0;           // every weight stage of the layer stays in shared memory

  const ConvGeom& g = p.g;
  const int tiles_per_img = g.tiles_x * g.tiles_y;
  const int num_tiles = g.n_img * tiles_per_img;
  const int groups = (num_tiles + 1) >> 1;
  const int num_items = groups * p.n_tiles;
  const int cluster_id = blockIdx.x >> 1;
  const int num_clusters = gridDim.x >> 1;
  const int nseg = p.h2_nseg;                         // fp32-promotion segments per tile (same rule as seg_end below)
  const int nslots = nseg + (NPLANES == 2 ? 1 : 0);   // accumulation slots (= promotions) per tile

  if (warp < kEpiWarp0) {
    ptx::setmaxnreg_dec<kRegsIssue>();   // 168 x 384 registers at launch = 128 x 40 + 256 x 232: a larger issue budget would leave setmaxnreg.inc waiting forever
    if (warp == 0) {
      // ============================== TMA producer: A boxes (both CTAs) ==============================
      if (lane == 0) {
        ptx::prefetch_tensormap(&tm_hi);
        if (NPLANES == 2) ptx::prefetch_tensormap(&tm_lo);
        int a = 0;
        uint32_t pha = 0;
        for (int item = cluster_id; item < num_items; item += num_clusters) {
          int tile = (item / p.n_tiles) * 2 + (int)rank;
          if (tile >= num_tiles) tile = num_tiles - 1;       // lockstep filler (stores are masked)
          const int img = tile / tiles_per_img;
          const int t2 = tile - img * tiles_per_img;
          const int ty = t2 / g.tiles_x, tx = t2 - ty * g.tiles_x;
          for (int ch = 0; ch < p.chunks; ++ch) {
            ptx::mbar_wait(&a_empty[a], pha ^ 1);
            uint8_t* slot = smem_a + (size_t)a * A_SLOT;
            const uint32_t lead = ptx::mapa_shared(ptx::smem_u32(&a_full[a]), 0);
            if (leader) ptx::mbar_arrive_expect_tx(&a_full[a], (uint32_t)(2 * NPLANES * kHalo1Rows * 128));
            ptx::tma_load_4d_2sm(slot, &tm_hi, lead, ch * KC, tx * kHaloTW - 1, ty * kHaloTH - 1, img);
            if (NPLANES == 2)
              ptx::tma_load_4d_2sm(slot + AH_BYTES, &tm_lo, lead, ch * KC, tx * kHaloTW - 1, ty * kHaloTH - 1, img);
            if (++a == num_a) { a = 0; pha ^= 1; }
          }
        }
      }
    } else if (warp == 2) {
      // ============================== TMA producer: weight halves (both CTAs) ==============================
      if (lane == 0) {
        ptx::prefetch_tensormap(&tm_w);
        const int wrows = NPLANES * half_rows;               // rows of one (tile, rank) block in the packed weights
        int b = 0;
        uint32_t phb = 0;
        for (int item = cluster_id; item < num_items; item += num_clusters) {
          const int n_tile = item % p.n_tiles;
          if (resident && item != cluster_id) break;          // loaded once, used by every tile of this CTA
          for (int st = 0; st < nst; ++st) {
            ptx::mbar_wait(&b_empty[b], phb ^ 1);
            const uint32_t lead = ptx::mapa_shared(ptx::smem_u32(&b_full[b]), 0);
            if (leader) ptx::mbar_arrive_expect_tx(&b_full[b], (uint32_t)(2 * B_STAGE));
            const int wblock = ((n_tile * nst + st) * 2 + (int)rank);
            ptx::tma_load_2d_2sm(smem_b + (size_t)b * B_STAGE, &tm_w, lead, 0, wblock * wrows);
            if (++b == num_b) { b = 0; phb ^= 1; }
          }
        }
      }
    } else if (warp == 1 && leader) {
      // ============================== MMA issuer (leader CTA only) ================================
      const uint32_t idesc = (1u << 4) | ((uint32_t)(p.n_pad >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
      const uint32_t sa_u32 = ptx::smem_u32(smem_a), sb_u32 = ptx::smem_u32(smem_b);
      int sa = 0, sb = 0;
      uint32_t spa = 0, spb = 0;
      // Accumulation slots rotate over the nbuf TMEM buffers: bd = buffer of the current dominant slot, bc = the next one;
      // bit b of `phm` = completed uses of buffer b mod 2 (mbarrier phase parity).  Plain increments and selects instead
      // of slot % nbuf keep all of it in uniform registers.
      uint32_t bd = 0, bc = 0, phm = 0;
      const int seg_target = 12 * p.seg_chunks;             // promotion period in 16-channel slices (12 = one full (chunk, dx) unit)
#ifdef DCSCN_H2_DEBUG
      long long w_a = 0, w_b = 0, w_acc = 0;
      const long long t_begin = clock64();
#endif
      for (int item = cluster_id; item < num_items; item += num_clusters) {
        { H2_T0(); ptx::mbar_wait(&acc_empty[bd], ((phm >> bd) & 1u) ^ 1u); H2_ACC(w_acc); }   // takes the dominant products of segment 0
        int s = 0;                                          // segment of the tile
        int dom = 0;                                        // stage weight issued into the open segment (12 per unit)
        bool seg_open = true;
        uint32_t tmem_d = 0, tmem_c = 0, acc_d0 = 0;
        bool fresh = true;                                  // the next UMMA slice opens the segment's accumulation slots
        int st = 0;                                         // weight stage of the item

        // one stage per tap, taps in (dx, dy) order, dy unrolled
        for (int ch = 0; ch < p.chunks; ++ch) {
          const int kt = min(4, (p.cin_pad - (ch << 6)) >> 4);      // 16-channel slices per tap (3 in a 48-channel tail)
          { H2_T0(); ptx::mbar_wait(&a_full[sa], spa); H2_ACC(w_a); }   // the chunk's halo box serves all nine taps
          // low descriptor word (start address >> 4 | LBO) of the A slot's hi plane; slots are 1024-byte aligned
          const uint32_t a_desc0 = (((sa_u32 + (uint32_t)sa * (uint32_t)A_SLOT) & 0x3FFFFu) >> 4) | (1u << 16);
          for (int dx = 0; dx < 3; ++dx) {
            if (seg_open) {
              bc = (bd + 1u == nbuf) ? 0u : bd + 1u;
              if (NPLANES == 2) { H2_T0(); ptx::mbar_wait(&acc_empty[bc], ((phm >> bc) & 1u) ^ 1u); H2_ACC(w_acc); }
              tmem_d = tmem_base + bd * (uint32_t)acc_stride;
              tmem_c = tmem_base + bc * (uint32_t)acc_stride;
              fresh = true;
              acc_d0 = (NPLANES == 2 && s > 0) ? 1u : 0u;     // the dominant slot already holds the previous corrections
              seg_open = false;
            }
            dom += 12;
            const bool seg_end = (dom >= seg_target) || (st + 3 == nst);   // same rule as h2_segments in engine.cu
#pragma unroll
            for (int dy = 0; dy < 3; ++dy, ++st) {
              if (!resident || item == cluster_id) { H2_T0(); ptx::mbar_wait(&b_full[sb], spb); H2_ACC(w_b); }   // resident stages landed during the first item
              ptx::tc_fence_after();
              const uint32_t b_addr = sb_u32 + (uint32_t)sb * (uint32_t)B_STAGE;
              uint32_t bh = desc_lo_t<KC>(b_addr), bl = desc_lo_t<KC>(b_addr + BH_BYTES);
              uint32_t ah = a_desc0 + (uint32_t)(dy * kHalo1W + dx) * 8u;
              uint32_t al = ah + (uint32_t)(AH_BYTES >> 4);
              if (ptx::elect_one()) {
                constexpr uint32_t kDescHiA = (uint32_t)((kHalo1W * 128) >> 4) | (1u << 14) | (2u << 29);   // SBO 1280, SW128, base offset 0
                constexpr uint32_t kDescHiB = (uint32_t)(TcSmem<KC>::kSbo >> 4) | (1u << 14) | ((uint32_t)TcSmem<KC>::kLayout << 29);
                // slice 0 may open the segment's accumulation slots; slices 1.. always accumulate.  Full chunks (kt == 4)
                // run the remaining slices as straight-line code: the single issuing thread spends ~7 instructions per
                // slice instead of ~20 (loop control + vector->uniform moves), which is what bounds the thin layers
                // (N <= 64: a UMMA lasts 24-32 cycles).
                {
                  const uint64_t da_hi = ((uint64_t)kDescHiA << 32) | ah, db_hi = ((uint64_t)kDescHiB << 32) | bh;
                  if (fresh) {
                    if (NPLANES == 2) {
                      ptx::mma_f16_ss_2sm(tmem_c, ((uint64_t)kDescHiA << 32) | al, db_hi, idesc, 0);
                      ptx::mma_f16_ss_2sm_acc(tmem_c, da_hi, ((uint64_t)kDescHiB << 32) | bl, idesc);
                    }
                    ptx::mma_f16_ss_2sm(tmem_d, da_hi, db_hi, idesc, acc_d0);
                  } else {
                    if (NPLANES == 2) {
                      ptx::mma_f16_ss_2sm_acc(tmem_c, ((uint64_t)kDescHiA << 32) | al, db_hi, idesc);
                      ptx::mma_f16_ss_2sm_acc(tmem_c, da_hi, ((uint64_t)kDescHiB << 32) | bl, idesc);
                    }
                    ptx::mma_f16_ss_2sm_acc(tmem_d, da_hi, db_hi, idesc);
                  }
                }
                // slices 1 .. kt - 1 as straight-line code for EVERY kt: almost every layer ends in a 16 / 32 / 48-channel tail
                // chunk (kt = 1 / 2 / 3), and a counted loop costs the single issuing thread ~20 instructions per slice
                // (loop control, vector -> uniform moves of the advancing descriptors) against ~7 here
#define H2_SLICE(KS)                                                                                                       \
  {                                                                                                                        \
    const uint64_t da_hi = ((uint64_t)kDescHiA << 32) | (ah + 2u * (KS)), db_hi = ((uint64_t)kDescHiB << 32) | (bh + 2u * (KS)); \
    if (NPLANES == 2) {                                                                                                    \
      ptx::mma_f16_ss_2sm_acc(tmem_c, ((uint64_t)kDescHiA << 32) | (al + 2u * (KS)), db_hi, idesc);                       \
      ptx::mma_f16_ss_2sm_acc(tmem_c, da_hi, ((uint64_t)kDescHiB << 32) | (bl + 2u * (KS)), idesc);                       \
    }                                                                                                                      \
    ptx::mma_f16_ss_2sm_acc(tmem_d, da_hi, db_hi, idesc);                                                                 \
  }
                if (kt >= 2) H2_SLICE(1)
                if (kt >= 3) H2_SLICE(2)
                if (kt == 4) H2_SLICE(3)
#undef H2_SLICE
                if (!resident) ptx::mma_commit_2sm(&b_empty[sb], 3);
                if (dy == 2 && dx == 2) ptx::mma_commit_2sm(&a_empty[sa], 3);
                if (dy == 2 && seg_end) {
                  ptx::mma_commit_2sm(&acc_full[bd], 3);
                  if (NPLANES == 2 && s == nseg - 1) ptx::mma_commit_2sm(&acc_full[bc], 3);
                }
              }
              fresh = false;
              __syncwarp();
              if (resident) {
                ++sb;                                             // stage st lives in ring slot st; phase 0 stays complete
              } else if (++sb == num_b) {
                sb = 0;
                spb ^= 1;
              }
            }
            if (seg_end) {
              ++s;
              dom = 0;
              seg_open = true;
              phm ^= 1u << bd;                                // this use of the dominant buffer is complete
              bd = bc;
            }
          }
          if (++sa == num_a) { sa = 0; spa ^= 1; }
        }
        if (NPLANES == 2) {                                         // the corrections-only slot of the last segment
          phm ^= 1u << bd;
          bd = (bd + 1u == nbuf) ? 0u : bd + 1u;
        }
        if (resident) sb = 0;
      }
#ifdef DCSCN_H2_DEBUG
      if (p.dbg != nullptr && lane == 0) {
        unsigned long long* d = p.dbg + (size_t)cluster_id * 8;
        d[0] = (unsigned long long)(clock64() - t_begin);
        d[1] = (unsigned long long)w_a;
        d[2] = (unsigned long long)w_b;
        d[3] = (unsigned long long)w_acc;
      }
#endif
    }
  } else {
    ptx::setmaxnreg_inc<kRegsEpilogue>();
    // ============================== epilogue (both CTAs, own 128 TMEM lanes) ==================================
    const int ew = warp - kEpiWarp0;
    const int quad = warp & 3;
    const int grp = ew >> 2;
    const int row = quad * 32 + lane;
    const int py = row / kHaloTW, px = row - py * kHaloTW;
    const int n_total = p.n_tiles * p.n_pad;
    const int nch = p.n_pad >> 4;
    const int per = (nch + kColSplit - 1) / kColSplit;
    const int first_chunk = grp * per;
    const int my_chunks = (nch - first_chunk) < per ? ((nch - first_chunk) > 0 ? nch - first_chunk : 0) : per;
    const int col_base = first_chunk * 16;
    const uint32_t lead_acc_empty0 = ptx::mapa_shared(ptx::smem_u32(&acc_empty[0]), 0);
    const uint32_t taddr0 = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)col_base;
    uint32_t eb = 0, ephm = 0;                           // buffer of the next slot to drain, per-buffer phase parity
#ifdef DCSCN_H2_DEBUG
    long long w_full = 0, t_store = 0;
    const long long t_begin = clock64();
#endif
    for (int item = cluster_id; item < num_items; item += num_clusters) {
      const int n_tile = item % p.n_tiles;
      const int tile = (item / p.n_tiles) * 2 + (int)rank;
      const bool real = tile < num_tiles;
      const int img = tile / tiles_per_img;
      const int t2 = tile - img * tiles_per_img;
      const int ty = t2 / g.tiles_x, tx = t2 - ty * g.tiles_x;
      const int y = ty * kHaloTH + py, x = tx * kHaloTW + px;
      const bool valid = real && (y < g.H) && (x < g.W);

      float sum[kMaxColChunks][16];
#pragma unroll
      for (int j = 0; j < kMaxColChunks; ++j)
#pragma unroll
        for (int i = 0; i < 16; ++i) sum[j][i] = 0.f;
      for (int s = 0; s < nslots; ++s) {
        const uint32_t buf = eb;
        { H2_T0(); ptx::mbar_wait(&acc_full[buf], (ephm >> buf) & 1u); H2_ACC(w_full); }
        ptx::tc_fence_after();
        const uint32_t taddr = taddr0 + buf * (uint32_t)acc_stride;
        // fp32 round-to-nearest promotion of the slot: wide TMEM loads (64 / 32 columns per instruction); columns
        // past this thread's share may be read (they stay inside the 512 allocated columns) but are never stored.
#pragma unroll
        for (int j = 0; j < kMaxColChunks; j += 4) {
          if (j < my_chunks) {
            if (my_chunks - j > 2) {
              float v[64];
              ptx::tmem_ld64(taddr + j * 16, v);
#pragma unroll
              for (int i = 0; i < 64; ++i) sum[j + (i >> 4)][i & 15] += v[i];
            } else {
              float v[32];
              ptx::tmem_ld32(taddr + j * 16, v);
#pragma unroll
              for (int i = 0; i < 32; ++i) sum[j + (i >> 4)][i & 15] += v[i];
            }
          }
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_cluster(lead_acc_empty0 + (uint32_t)(buf * sizeof(uint64_t)));
        ephm ^= 1u << buf;
        eb = (eb + 1u == nbuf) ? 0u : eb + 1u;
      }
      H2_T0();
      if (p.epi.mode == EPI_D2S_RDOT) {
        float v[9];
#pragma unroll
        for (int t = 0; t < 9; ++t) v[t] = 0.f;
        const int share = per * 16;                       // columns of one epilogue thread
#pragma unroll
        for (int j = 0; j < kMaxColChunks; ++j) {
          if (j < my_chunks) {
            const int cg = n_tile * p.n_pad + col_base + j * 16;
            if (cg < p.epi.n_valid) {
              const int ij = cg / p.epi.d2s_cout, c = cg - ij * p.epi.d2s_cout;
              rdot_accumulate16(p.epi, s_rdot, cg, c, sum[j], v);
              // flush when this thread has seen its whole part of the sub-pixel (all of it when rdot_parts == 1)
              const bool last = (p.epi.rdot_parts > 1) ? (j == my_chunks - 1) : (c + 16 == p.epi.d2s_cout);
              if (last && valid) rdot_flush(p.epi, g, img, y, x, ij, p.epi.rdot_parts > 1 ? c / share : 0, v);
            }
          }
        }
      } else if (p.epi.store_mode == 2 && p.epi.mode == EPI_PLANES && p.epi.num_seg == 1 && p.epi.seg[0].dst_zneg == nullptr) {
        // Lane-pair stores.  Lanes 2k and 2k + 1 hold two horizontally adjacent pixels; for every PAIR of 16-column chunks
        // they swap halves, so that one store instruction writes chunk j (even lane) and chunk j + 1 (odd lane) of the SAME
        // pixel - 64 contiguous bytes, one 128-byte line per two lanes instead of one per lane.  All lanes take part in the
        // shuffles; stores are predicated on the pixel they write.
        const EpiSegment sg = p.epi.seg[0];
        const bool odd = (lane & 1) != 0;
        const bool pvalid = __shfl_xor_sync(0xffffffffu, valid ? 1 : 0, 1) != 0;
        const bool valid_e = odd ? pvalid : valid, valid_o = odd ? valid : pvalid;   // the pair's even / odd pixel
        const size_t pix = (size_t)((size_t)img * g.H + y) * g.W + x;
        const size_t pix_e = odd ? pix - 1 : pix, pix_o = odd ? pix : pix + 1;
        // (training forwards, which also store min(z, 0), take the per-lane path below)
#pragma unroll
        for (int j = 0; j < kMaxColChunks; j += 2) {
          if (j + 1 < my_chunks) {
            const int cg0 = n_tile * p.n_pad + col_base + j * 16;
            float v0[16], v1[16];
            uint32_t zdummy[8];
            epilogue_values16(p.epi, g, n_total, img, y, x, cg0, sum[j], v0, zdummy, false);
            epilogue_values16(p.epi, g, n_total, img, y, x, cg0 + 16, sum[j + 1], v1, zdummy, false);
            const int colA = (cg0 - sg.col_begin) + (odd ? 16 : 0);        // this lane's column in both stores
            const size_t offA = pix_e * sg.pitch + colA, offB = pix_o * sg.pitch + colA;
            if (cg0 >= sg.col_begin && cg0 + 16 < sg.col_end) {
              // one plane at a time (hi, then lo) keeps the live registers of the exchange small
#pragma unroll
              for (int pln = 0; pln < 2; ++pln) {
                __half* dstp = pln == 0 ? sg.dst_hi : sg.dst_lo;
                if (dstp == nullptr) continue;
                uint32_t w0[8], w1[8];                                      // this plane's packed words of chunk j / j + 1
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  uint32_t hh, ll;
                  split_f16x2(v0[2 * i], v0[2 * i + 1], hh, ll);
                  w0[i] = pln == 0 ? hh : ll;
                  split_f16x2(v1[2 * i], v1[2 * i + 1], hh, ll);
                  w1[i] = pln == 0 ? hh : ll;
                }
                // even lane: keeps chunk j, sends chunk j + 1, receives the odd pixel's chunk j;
                // odd lane:  keeps chunk j + 1, sends chunk j, receives the even pixel's chunk j + 1
                uint32_t wa[8], wb[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  const uint32_t r = __shfl_xor_sync(0xffffffffu, odd ? w0[i] : w1[i], 1);
                  wa[i] = odd ? r : w0[i];        // the even pixel: own chunk j (even lane) | received chunk j + 1 (odd lane)
                  wb[i] = odd ? w1[i] : r;        // the odd pixel: received chunk j (even lane) | own chunk j + 1 (odd lane)
                }
                if (valid_e) stg256(dstp + offA, wa);
                if (valid_o) stg256(dstp + offB, wb);
              }
            } else if (valid) {                  // a pair that straddles the segment's end: plain per-lane stores
              epilogue_store16(p.epi, g, n_total, img, y, x, cg0, sum[j]);
              epilogue_store16(p.epi, g, n_total, img, y, x, cg0 + 16, sum[j + 1]);
            }
          } else if (j < my_chunks && valid) {
            epilogue_store16(p.epi, g, n_total, img, y, x, n_tile * p.n_pad + col_base + j * 16, sum[j]);
          }
        }
      } else if (valid) {
#pragma unroll
        for (int j = 0; j < kMaxColChunks; ++j)
          if (j < my_chunks) epilogue_store16(p.epi, g, n_total, img, y, x, n_tile * p.n_pad + col_base + j * 16, sum[j]);
      }
      H2_ACC(t_store);
    }
#ifdef DCSCN_H2_DEBUG
    if (p.dbg != nullptr && leader && warp == kEpiWarp0 && lane == 0) {
      unsigned long long* d = p.dbg + (size_t)cluster_id * 8;
      d[4] = (unsigned long long)(clock64() - t_begin);
      d[5] = (unsigned long long)w_full;
      d[6] = (unsigned long long)t_store;
    }
#endif
  }

  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc_2sm(tmem_base, 512);
  }
}

}  // namespace dcscn
