// CTA-pair tcgen05 implicit-GEMM convolution (see conv_tc.cuh for what the tensor-core kernels share).
//
// Measured on B200 (profiles/r1a_*): a single-CTA form of this kernel was bound by bytes entering each SM (TMA -> shared
// memory, ~28 B/clk/SM) - every 128-pixel tile streams the whole layer's weight tiles - not by the tensor pipe (25 % active).
// Here two CTAs of one TPC form a cluster and issue `tcgen05.mma.cta_group::2` with M = 256 (two 128-pixel tiles):
// each CTA stages only HALF of every weight tile (N/2 rows) and the tensor core reads the other half from the
// peer's shared memory, so weight bytes per SM (and weight shared-memory reads) are halved.
//   * rank 0 ("leader") issues all UMMAs; both CTAs run a TMA producer for their own pixel tile + weight half,
//     completing transactions on the LEADER's `full` barrier (cp.async.bulk.tensor ... .cta_group::2);
//   * tcgen05.commit.cta_group::2 ... .multicast::cluster releases pipeline stages / publishes accumulator segments
//     to both CTAs; both CTAs' epilogue warps promote their own 128 TMEM lanes and release the accumulator on the
//     leader's barrier (remote mbarrier arrive).
#pragma once
#include "conv_tc.cuh"

namespace dcscn {

namespace ptx {

__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(cta_rank));
  return r;
}
// Arrival on an mbarrier of (possibly) the peer CTA.  RELAXED on purpose: the callers are epilogue warps handing a TMEM
// accumulator back to the MMA issuer after `tcgen05.wait::ld` + `tcgen05.fence::before_thread_sync` - the values are in
// registers, there is nothing in memory to publish.  The default `.release.cluster` form costs a MEMBAR.ALL.GPU + ERRBAR
// per arrival (it waits for the epilogue's own outstanding global stores): ncu showed 20 % of all epilogue-warp stall
// samples there and the MMA issuer parked on acc_empty (profiles/r2b_*).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA loads whose completion is signalled on an mbarrier that may live in the peer CTA of the pair.
__device__ __forceinline__ void tma_load_4d_2sm(void* smem_dst, const CUtensorMap* tm, uint32_t bar_cluster_addr, int c0,
                                                int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* tm, uint32_t bar_cluster_addr, int c0,
                                                int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* smem_result, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "r"(cols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2sm() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void mma_f16_ss_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same with the accumulate input always enabled (no runtime predicate to materialise in front of the instruction).
__device__ __forceinline__ void mma_f16_ss_2sm_acc(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.eq.u32 p, 1, 1;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc)
      : "memory");
}
__device__ __forceinline__ void mma_commit_2sm(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}

}  // namespace ptx

__host__ __device__ inline size_t tc_pair_stage_bytes(int nplanes, int n_pad) {
  return (size_t)nplanes * ((size_t)kTileM * 64 * 2 + (size_t)(n_pad / 2) * 64 * 2);
}

constexpr int kPairAccBars = 4;          // accumulation barriers (two-pass mode uses 2, streaming mode 4 TMEM buffers)
constexpr int kPairStreamStride = 128;   // TMEM columns between the four buffers of the streaming mode (n_pad <= 128)
constexpr int kPairBarBytes = 512;       // barrier block in front of the R-CNN weight staging area

// p.pair_stream != 0 (1x1 layers, NPLANES == 2, n_pad <= 128): the streaming accumulation of conv_tc_halo2.cuh - the
// correction products of segment s go to slot s + 1 FIRST, the dominant products to slot s, slots rotate over four
// TMEM buffers - so every stage is released by the commit behind its own UMMAs and the whole ring is prefetch depth.
// A1|B1 reads 3.1 GB of concatenated features per 256-tile step: it is bound by HBM, and the two-pass form kept
// seg_chunks of its five 44 KB stages parked until their second pass.
template <int NPLANES>
__global__ void __launch_bounds__(kTcThreads, 1)
conv_tc_pair_kernel(const __grid_constant__ CUtensorMap tm_hi, const __grid_constant__ CUtensorMap tm_lo,
                    const __grid_constant__ CUtensorMap tm_w, const ConvTCParams p, const int num_stages) {
  constexpr int KC = 64;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int A_BYTES = TcSmem<KC>::kABytes;
  const int half_rows = p.n_pad >> 1;                 // weight-tile rows staged by each CTA of the pair
  const int BH_BYTES = half_rows * KC * 2;            // one plane of this CTA's weight half
  const int STAGE_BYTES = NPLANES * (A_BYTES + BH_BYTES);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)num_stages * STAGE_BYTES);
  uint64_t* empty_bar = full_bar + kMaxStages;
  uint64_t* acc_full = empty_bar + kMaxStages;
  uint64_t* acc_empty = acc_full + kPairAccBars;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + kPairAccBars);
  float* s_rdot = reinterpret_cast<float*>(tmem_slot + 4);   // 16-byte aligned (barriers start 1024-aligned)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < num_stages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);                     // leader's producer arrive + both CTAs' TMA bytes
      ptx::mbar_init(&empty_bar[s], 1);                    // leader's tcgen05.commit (multicast to both CTAs)
    }
    for (int s = 0; s < kPairAccBars; ++s) {
      ptx::mbar_init(&acc_full[s], 1);                     // leader's tcgen05.commit (multicast)
      ptx::mbar_init(&acc_empty[s], 2 * kEpiWarps);        // epilogue warps of both CTAs (used on the leader only)
    }
    ptx::fence_barrier_init();
    ptx::fence_proxy_async();
  }
  if (warp == 1) {
    ptx::tmem_alloc_2sm(tmem_slot, kAccStages * kAccStride);
    ptx::tmem_relinquish_2sm();
  }
  if (p.epi.mode == EPI_D2S_RDOT)
    for (int i = threadIdx.x; i < p.epi.rdot_taps * p.epi.d2s_cout; i += blockDim.x) s_rdot[i] = p.epi.rdot_w[i];
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const ConvGeom& g = p.g;
  const int tiles_per_img = g.tiles_x * g.tiles_y;
  const int num_tiles = g.n_img * tiles_per_img;
  const int groups = (num_tiles + 1) >> 1;
  const int num_items = groups * p.n_tiles;
  const int cluster_id = blockIdx.x >> 1;
  const int num_clusters = gridDim.x >> 1;
  const int taps = p.ksz * p.ksz;
  const int half = p.ksz >> 1;
  const int total_chunks = taps * p.chunks;

  if (warp < kEpiWarp0) {
    ptx::setmaxnreg_dec<kRegsIssue>();
    if (warp == 0) {
      // ============================== TMA producer (both CTAs) ==============================
      if (lane == 0) {
        ptx::prefetch_tensormap(&tm_hi);
        if (NPLANES == 2) ptx::prefetch_tensormap(&tm_lo);
        ptx::prefetch_tensormap(&tm_w);
        const int wrows = NPLANES * half_rows;               // rows of one (tile, rank) block in the packed weights
        int stage = 0;
        uint32_t phase = 0;
        for (int item = cluster_id; item < num_items; item += num_clusters) {
          const int n_tile = item % p.n_tiles;
          int tile = (item / p.n_tiles) * 2 + (int)rank;
          if (tile >= num_tiles) tile = num_tiles - 1;       // lockstep filler (stores are masked)
          const int img = tile / tiles_per_img;
          const int t2 = tile - img * tiles_per_img;
          const int ty = t2 / g.tiles_x, tx = t2 - ty * g.tiles_x;
          for (int tap = 0; tap < taps; ++tap) {
            const int dy = tap / p.ksz - half, dx = tap % p.ksz - half;
            for (int ch = 0; ch < p.chunks; ++ch) {
              ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
              uint8_t* st = smem + (size_t)stage * STAGE_BYTES;
              const uint32_t lead_full = ptx::mapa_shared(ptx::smem_u32(&full_bar[stage]), 0);
              if (leader) ptx::mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)(2 * STAGE_BYTES));
              ptx::tma_load_4d_2sm(st, &tm_hi, lead_full, ch * KC, tx * g.TW + dx, ty * g.TH + dy, img);
              if (NPLANES == 2)
                ptx::tma_load_4d_2sm(st + A_BYTES, &tm_lo, lead_full, ch * KC, tx * g.TW + dx, ty * g.TH + dy, img);
              const int wblock = ((n_tile * taps + tap) * p.chunks + ch) * 2 + (int)rank;
              ptx::tma_load_2d_2sm(st + NPLANES * A_BYTES, &tm_w, lead_full, 0, wblock * wrows);
              if (++stage == num_stages) { stage = 0; phase ^= 1; }
            }
          }
        }
      }
    } else if (warp == 1 && leader) {
      // ============================== MMA issuer (leader CTA only) ================================
      const uint32_t idesc = (1u << 4) | ((uint32_t)(p.n_pad >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
      const uint32_t smem_base_u32 = ptx::smem_u32(smem);
      int stage = 0;
      uint32_t phase = 0;
      uint32_t seg_count = 0;
      if (NPLANES == 2 && p.pair_stream) {
        uint32_t bd = 0, phm = 0;                            // dominant buffer of the open segment, per-buffer phase bits
        for (int item = cluster_id; item < num_items; item += num_clusters) {
          ptx::mbar_wait(&acc_empty[bd], ((phm >> bd) & 1u) ^ 1u);
          for (int c0 = 0; c0 < total_chunks; c0 += p.seg_chunks) {
            const uint32_t bc = (bd + 1u) & 3u;
            ptx::mbar_wait(&acc_empty[bc], ((phm >> bc) & 1u) ^ 1u);
            ptx::tc_fence_after();
            const uint32_t tmem_d = tmem_base + bd * (uint32_t)kPairStreamStride;
            const uint32_t tmem_c = tmem_base + bc * (uint32_t)kPairStreamStride;
            uint32_t acc_c = 0;                              // corrections open their slot
            uint32_t acc_d = c0 > 0 ? 1u : 0u;               // the dominant slot already holds the previous corrections
            const int c1 = (c0 + p.seg_chunks < total_chunks) ? c0 + p.seg_chunks : total_chunks;
            for (int c = c0; c < c1; ++c) {
              const int ch = c % p.chunks;
              ptx::mbar_wait(&full_bar[stage], phase);
              ptx::tc_fence_after();
              const uint32_t st_addr = smem_base_u32 + (uint32_t)stage * (uint32_t)STAGE_BYTES;
              uint32_t ah = desc_lo_t<KC>(st_addr), al = desc_lo_t<KC>(st_addr + A_BYTES);
              uint32_t bh = desc_lo_t<KC>(st_addr + NPLANES * A_BYTES), bl = desc_lo_t<KC>(st_addr + NPLANES * A_BYTES + BH_BYTES);
              int ksteps = (p.cin_pad - ch * KC);
              ksteps = (ksteps > KC ? KC : ksteps) >> 4;
              if (ptx::elect_one()) {
#pragma unroll 1
                for (int ks = 0; ks < ksteps; ++ks) {
                  ptx::mma_f16_ss_2sm(tmem_c, make_desc64_t<KC>(al), make_desc64_t<KC>(bh), idesc, acc_c);
                  ptx::mma_f16_ss_2sm_acc(tmem_c, make_desc64_t<KC>(ah), make_desc64_t<KC>(bl), idesc);
                  ptx::mma_f16_ss_2sm(tmem_d, make_desc64_t<KC>(ah), make_desc64_t<KC>(bh), idesc, acc_d);
                  acc_c = 1;
                  acc_d = 1;
                  ah += 2; al += 2; bh += 2; bl += 2;       // 32 bytes (16 fp16 along K) in 16-byte descriptor units
                }
                ptx::mma_commit_2sm(&empty_bar[stage], 3);   // the stage is free once these UMMAs have read it
                if (c == c1 - 1) {
                  ptx::mma_commit_2sm(&acc_full[bd], 3);
                  if (c1 == total_chunks) ptx::mma_commit_2sm(&acc_full[bc], 3);   // corrections-only slot of the last segment
                }
              }
              acc_c = 1;
              acc_d = 1;
              __syncwarp();
              if (++stage == num_stages) { stage = 0; phase ^= 1; }
            }
            phm ^= 1u << bd;
            bd = bc;
          }
          phm ^= 1u << bd;                                   // the corrections-only slot
          bd = (bd + 1u) & 3u;
        }
      } else
      for (int item = cluster_id; item < num_items; item += num_clusters) {
        for (int c0 = 0; c0 < total_chunks; c0 += p.seg_chunks) {
          const int acc = seg_count & 1;
          ptx::mbar_wait(&acc_empty[acc], ((seg_count >> 1) & 1) ^ 1);
          ptx::tc_fence_after();
          const uint32_t tmem_d = tmem_base + (uint32_t)(acc * kAccStride);
          uint32_t accumulate = 0;
          const int c1 = (c0 + p.seg_chunks < total_chunks) ? c0 + p.seg_chunks : total_chunks;
          // Pass A: as the stages of this segment land, issue the small correction products (a_lo*w_hi, a_hi*w_lo).
          // Pass B: the dominant a_hi*w_hi products, releasing each stage.  The accumulator only becomes large in
          // pass B, so only those UMMAs contribute truncation error: 3x fewer "effective" steps per segment.
          // Warp-uniform descriptor arithmetic; only the UMMA / commit instructions are single-lane (elect.sync), which
          // keeps the issue loop on the uniform datapath.
          int st = stage;
          uint32_t ph = phase;
          for (int c = c0; c < c1; ++c) {
            const int ch = c % p.chunks;
            ptx::mbar_wait(&full_bar[st], ph);
            ptx::tc_fence_after();
            if (NPLANES == 2) {
              const uint32_t st_addr = smem_base_u32 + (uint32_t)st * (uint32_t)STAGE_BYTES;
              const uint32_t la_hi = desc_lo_t<KC>(st_addr);
              const uint32_t la_lo = desc_lo_t<KC>(st_addr + A_BYTES);
              const uint32_t lb_hi = desc_lo_t<KC>(st_addr + NPLANES * A_BYTES);
              const uint32_t lb_lo = desc_lo_t<KC>(st_addr + NPLANES * A_BYTES + BH_BYTES);
              int ksteps = (p.cin_pad - ch * KC);
              ksteps = (ksteps > KC ? KC : ksteps) >> 4;
              if (ptx::elect_one()) {
#pragma unroll 1
                for (int ks = 0; ks < ksteps; ++ks) {
                  const uint32_t kadd = (uint32_t)ks * 2u;  // 32 bytes (16 fp16 along K) in 16-byte descriptor units
                  ptx::mma_f16_ss_2sm(tmem_d, make_desc64_t<KC>(la_lo + kadd), make_desc64_t<KC>(lb_hi + kadd), idesc, accumulate);
                  ptx::mma_f16_ss_2sm(tmem_d, make_desc64_t<KC>(la_hi + kadd), make_desc64_t<KC>(lb_lo + kadd), idesc, 1);
                  accumulate = 1;
                }
              }
              accumulate = 1;
              __syncwarp();
            }
            if (++st == num_stages) { st = 0; ph ^= 1; }
          }
          st = stage;
          for (int c = c0; c < c1; ++c) {
            const int ch = c % p.chunks;
            const uint32_t st_addr = smem_base_u32 + (uint32_t)st * (uint32_t)STAGE_BYTES;
            const uint32_t la_hi = desc_lo_t<KC>(st_addr);
            const uint32_t lb_hi = desc_lo_t<KC>(st_addr + NPLANES * A_BYTES);
            int ksteps = (p.cin_pad - ch * KC);
            ksteps = (ksteps > KC ? KC : ksteps) >> 4;
            if (ptx::elect_one()) {
#pragma unroll 1
              for (int ks = 0; ks < ksteps; ++ks) {
                const uint32_t kadd = (uint32_t)ks * 2u;
                ptx::mma_f16_ss_2sm(tmem_d, make_desc64_t<KC>(la_hi + kadd), make_desc64_t<KC>(lb_hi + kadd), idesc, accumulate);
                accumulate = 1;
              }
              ptx::mma_commit_2sm(&empty_bar[st], 3);  // frees this smem stage once the UMMAs have read it
            }
            accumulate = 1;
            __syncwarp();
            if (++st == num_stages) st = 0;
          }
          stage = st;
          phase = ph;
          if (ptx::elect_one()) ptx::mma_commit_2sm(&acc_full[acc], 3);  // segment complete in both CTAs' TMEM
          __syncwarp();
          ++seg_count;
        }
      }
    }
  } else {
    ptx::setmaxnreg_inc<kRegsEpilogue>();
    // ============================== epilogue (both CTAs, own 128 TMEM lanes) ==================================
    const int ew = warp - kEpiWarp0;
    const int quad = warp & 3;
    const int grp = ew >> 2;
    const int row = quad * 32 + lane;
    const int py = row / g.TW, px = row - py * g.TW;
    const int n_total = p.n_tiles * p.n_pad;
    const int nch = p.n_pad >> 4;
    const int per = (nch + kColSplit - 1) / kColSplit;
    const int first_chunk = grp * per;
    const int my_chunks = (nch - first_chunk) < per ? ((nch - first_chunk) > 0 ? nch - first_chunk : 0) : per;
    const int col_base = first_chunk * 16;
    const bool stream = NPLANES == 2 && p.pair_stream != 0;
    const int nseg = (total_chunks + p.seg_chunks - 1) / p.seg_chunks + (stream ? 1 : 0);   // accumulation slots to drain
    const uint32_t lead_acc_empty0 = ptx::mapa_shared(ptx::smem_u32(&acc_empty[0]), 0);
    const uint32_t taddr0 = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)col_base;
    const uint32_t acc_mask = stream ? 3u : 1u, acc_stride = stream ? (uint32_t)kPairStreamStride : (uint32_t)kAccStride;
    const int acc_shift = stream ? 2 : 1;
    uint32_t seg_count = 0;
    for (int item = cluster_id; item < num_items; item += num_clusters) {
      const int n_tile = item % p.n_tiles;
      const int tile = (item / p.n_tiles) * 2 + (int)rank;
      const bool real = tile < num_tiles;
      const int img = tile / tiles_per_img;
      const int t2 = tile - img * tiles_per_img;
      const int ty = t2 / g.tiles_x, tx = t2 - ty * g.tiles_x;
      const int y = ty * g.TH + py, x = tx * g.TW + px;
      const bool valid = real && (y < g.H) && (x < g.W);

      float sum[kMaxColChunks][16];
#pragma unroll
      for (int j = 0; j < kMaxColChunks; ++j)
#pragma unroll
        for (int i = 0; i < 16; ++i) sum[j][i] = 0.f;
      for (int s = 0; s < nseg; ++s) {
        const uint32_t acc = seg_count & acc_mask;          // slots use the buffers round-robin in both modes
        ptx::mbar_wait(&acc_full[acc], (seg_count >> acc_shift) & 1);
        ptx::tc_fence_after();
        const uint32_t taddr = taddr0 + acc * acc_stride;
        // fp32 round-to-nearest promotion of the segment: wide TMEM loads (64 / 32 columns per instruction); columns
        // past this thread's share may be read (they stay inside the allocated columns) but are never stored.
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
        if (lane == 0) ptx::mbar_arrive_cluster(lead_acc_empty0 + (uint32_t)(acc * sizeof(uint64_t)));
        ++seg_count;
      }
      if (p.epi.mode == EPI_D2S_RDOT) {
        float v[9];
#pragma unroll
        for (int t = 0; t < 9; ++t) v[t] = 0.f;
#pragma unroll
        for (int j = 0; j < kMaxColChunks; ++j) {
          if (j < my_chunks) {
            const int cg = n_tile * p.n_pad + col_base + j * 16;
            if (cg < p.epi.n_valid) {
              const int ij = cg / p.epi.d2s_cout, c = cg - ij * p.epi.d2s_cout;
              rdot_accumulate16(p.epi, s_rdot, cg, c, sum[j], v);
              if (c + 16 == p.epi.d2s_cout && valid) rdot_flush(p.epi, g, img, y, x, ij, v);
            }
          }
        }
      } else if (valid) {
#pragma unroll
        for (int j = 0; j < kMaxColChunks; ++j)
          if (j < my_chunks) epilogue_store16(p.epi, g, n_total, img, y, x, n_tile * p.n_pad + col_base + j * 16, sum[j]);
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc_2sm(tmem_base, kAccStages * kAccStride);
  }
}

}  // namespace dcscn
