// The 3x3 convs (features[6..17], reference hardnet/HardNet.py:287-298) as persistent, warp-specialised tcgen05 implicit
// GEMMs: M = 128 output pixels per tile, N = C_out, K = 9 taps x C_in, cut into "k-blocks" of one tap x <=64 channels.
// Activations live in global memory CHANNEL-PLANAR: [patch][plane = c / 8][y][x][c % 8] (16 B per pixel and plane; stride-2
// consumers get the four row/column parity sub-planes [plane][ypar][xpar][y/2][x/2][8]). The A tile of a k-block is ONE 4-D
// TMA box (x * 8, y, patch, plane) whose start coordinate carries the tap shift; out-of-range x / y are zero-filled by TMA,
// which is exactly the conv's zero padding, and because x / y are per-patch tensor dimensions nothing bleeds between
// patches. The box lands in shared memory as [plane][pixel][8 channels], which is the UMMA no-swizzle K-major layout (core
// matrix = 8 pixels x 16 B, SBO = 128 B, LBO = plane pitch). The planar layout is what makes the epilogue's stores
// coalesce: a warp writes 32 pixels x 16 B = 512 contiguous bytes per instruction (NHWC rows would touch 32 cache lines).
//
// Two CTAs of one cluster (= the two SMs of a TPC) run tcgen05.mma.cta_group::2 with M = 256: each CTA owns one
// 128-pixel tile (A operand + accumulator in its own shared memory / TMEM) and HALF of the weight rows (B operand,
// C_out / 2 output channels), and the tensor cores of both SMs read B from both halves.
//
// Why: an SS-mode UMMA with M = 128 reads 4 KB of A and N * 32 B of B from shared memory per K = 16 step, and the
// shared-memory port moves 128 B/clk. At N = 128 that is 64 wavefronts for 64 clk of math - the port is saturated by
// the tensor core alone and every TMA write or epilogue access stalls it. In a pair each SM reads A (32 wavefronts)
// + half of B (N / 8), i.e. 48 per 64 clk at N = 128, and the weights of a layer fit in shared memory
// (conv6: 2 x 144 KB) so they are loaded once per CTA instead of streamed per tile.
//
// Protocol (a ring of A tiles and two accumulator buffers in TMEM, so the epilogue of tile i overlaps the MMAs of tile i+1;
// warp 0 = TMA producer, warp 1 = TMEM owner + UMMA issuer, warps 2..5 = epilogue):
//   * every CTA's TMA loads land in its own shared memory but complete_tx on the LEADER's (cluster rank 0) full
//     barrier (cp.async.bulk.tensor ... .cta_group::2), which counts one arrive.expect_tx from each producer;
//   * only the leader issues MMAs; tcgen05.commit ... .multicast::cluster frees the ring slot / publishes the
//     accumulator in both CTAs;
//   * both CTAs' epilogue warps release the accumulator on the leader's barrier (remote mbarrier.arrive).
#pragma once

#include "common.cuh"
#include "tc_conv.cuh"

namespace hn {

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> shared::cluster address of the same offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_cluster(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
  // default semantics (release at CTA scope): a cluster-scope release costs a MEMBAR.ALL.GPU per arrive
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx_cluster(uint32_t cluster_bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;" ::"r"(cluster_bar), "r"(bytes)
               : "memory");
}
// TMA loads whose completion is signalled on a barrier that may live in the peer CTA of the pair
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* tm, uint32_t cluster_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(cluster_bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(uint32_t dst, const CUtensorMap* tm, uint32_t cluster_bar, int c0, int c1,
                                                 int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(cluster_bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_f16_pair_w(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                                uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// kind::f8f6f4 twin (UTCQMMA.2CTA), see umma_f8_w
__device__ __forceinline__ void umma_f8_pair_w(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                               uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], da, db, %5, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrives on the barrier at this shared-memory offset in BOTH CTAs once the previously issued MMAs have retired.
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"(static_cast<uint16_t>(3))
               : "memory");
}

// ROWSHIFT (stride-1 layers): one TMA load per (kx, channel chunk) fetches the tile's band of image rows plus one
// halo row above and below; the three ky taps then read that SAME shared-memory tile through UMMA descriptors whose
// start address is advanced by ky image rows (whole 8-row core matrices). Cuts the L2->SMEM operand traffic from 9x
// to 3x(R+2)/R. When a tile spans several small patches (8x8 images: two patches) the box is ordered
// (x, patch, y, plane), so that shared memory holds [plane][y][patch][x] and a ky shift is still one uniform offset;
// the tile's M rows are then ordered (y, patch, x).
template <int CIN, int COUT, int HOUT, int STRIDE, int STAGES, bool ROWSHIFT, int KCB_ = 0>
struct PairCfg {
  static constexpr int KCB = KCB_ ? KCB_ : ((CIN >= 64) ? 128 : 64);   // bytes of one pixel's channel chunk
  static constexpr int KC = KCB / 2;                                   // channels per k-block
  static constexpr int CIN_CHUNKS = CIN / KC;
  static constexpr int KB = 9 * CIN_CHUNKS;                            // k-blocks per tile
  static constexpr int PIX = HOUT * HOUT;
  static constexpr int TILES_PER_PATCH = PIX >= kTileM ? PIX / kTileM : 0;
  static constexpr int ROWS_PER_TILE = PIX >= kTileM ? kTileM / HOUT : HOUT;
  static constexpr int PATCHES_PER_TILE = PIX >= kTileM ? 1 : kTileM / PIX;
  static constexpr int SPT = ROWSHIFT ? 3 * CIN_CHUNKS : KB;           // TMA loads of A (= pipeline stages) per tile
  static constexpr int NPL = KC / 8;                                   // 8-channel planes per k-block
  // one image row (of all the tile's patches when ROWSHIFT) inside one plane of the A tile
  static constexpr uint32_t ROW_BYTES = (ROWSHIFT ? PATCHES_PER_TILE : 1) * HOUT * 16;
  static constexpr uint32_t PLANE_BYTES = ROWSHIFT ? (ROWS_PER_TILE + 2) * ROW_BYTES : kTileM * 16;
  static constexpr uint32_t A_BYTES = NPL * PLANE_BYTES;
  static_assert(!ROWSHIFT || (STRIDE == 1 && ROW_BYTES % 128 == 0),
                "ROWSHIFT needs a stride-1 layer whose image rows are whole core matrices");
  static constexpr uint32_t BH_BYTES = (COUT / 2) * KCB;       // this CTA's half of one weight k-block
  static constexpr uint32_t W_BYTES = KB * BH_BYTES;           // resident half of the layer's weights
  static constexpr uint32_t STAGE_BYTES = A_BYTES;
  static constexpr uint32_t TMEM_COLS = tmem_cols_for(COUT);
  static constexpr size_t SMEM = size_t(W_BYTES) + size_t(STAGES) * STAGE_BYTES + 1024 + 256 + COUT * 4;
  static_assert(A_BYTES % 1024 == 0 && BH_BYTES % 1024 == 0, "swizzled weight tiles must stay 1024B aligned");
  static_assert(COUT % 32 == 0 && COUT <= 256, "cta_group::2 UMMA needs N % 16 == 0 and an even split of the rows");
  static_assert(SMEM <= 227 * 1024, "shared memory budget");
};

template <int CIN, int COUT, int HOUT, int STRIDE, int STAGES, bool ROWSHIFT, bool OUT_PARITY, int KCB_>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kTcThreads, 1)
conv3x3_pair_kernel(const __grid_constant__ TcParams p) {
  using C = PairCfg<CIN, COUT, HOUT, STRIDE, STAGES, ROWSHIFT, KCB_>;
  constexpr int N = COUT;
  constexpr int PPT = C::PATCHES_PER_TILE;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;   // identical in both CTAs (same kernel, same dynamic smem base)
  const uint32_t w_base = base;
  const uint32_t ring_base = base + C::W_BYTES;
  const uint32_t bar_base = ring_base + STAGES * C::STAGE_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };
  const uint32_t w_bar = bar_base + 8u * (2 * STAGES + 4);
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 5);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw_addr));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
  const int num_groups = (p.num_tiles + 1) / 2;   // a pass of the pair covers two consecutive tiles

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmA[0]);
    if (STRIDE == 2) {
      tma_prefetch_desc(&p.tmA[1]);
      tma_prefetch_desc(&p.tmA[2]);
      tma_prefetch_desc(&p.tmA[3]);
    }
    tma_prefetch_desc(&p.tmB);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < STAGES; ++s) {
        mbar_init(full_bar(s), 2);    // one arrive.expect_tx per CTA of the pair (only the leader's copy is used)
        mbar_init(empty_bar(s), 1);   // multicast tcgen05.commit
      }
      for (int a = 0; a < 2; ++a) {
        mbar_init(tfull_bar(a), 1);   // multicast tcgen05.commit
        mbar_init(tempty_bar(a), 8);  // four epilogue warps of each CTA (only the leader's copy is used)
      }
      mbar_init(w_bar, 2);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc_pair(tmem_slot, C::TMEM_COLS);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // the peer's barriers are initialised and its TMEM is allocated before anyone signals it
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ============================== TMA producer (both CTAs, warp-uniform) ==============================
    const uint32_t lead_w_bar = mapa_cluster(w_bar, 0);
    if (elect_one()) {
      mbar_arrive_expect_tx_cluster(lead_w_bar, C::W_BYTES);
#pragma unroll 1
      for (int kb = 0; kb < C::KB; ++kb)
        tma_load_2d_pair(w_base + kb * C::BH_BYTES, &p.tmB, lead_w_bar, kb * C::KC, static_cast<int>(rank) * (COUT / 2));
    }
    __syncwarp();
    int stage = 0;
    uint32_t phase = 0;
    for (int grp = pair; grp < num_groups; grp += num_pairs) {
      // tiles past the end of the batch read out-of-range patch coordinates: TMA zero-fills them
      const int tile = grp * 2 + static_cast<int>(rank);
      int patch0, y0;
      if (C::TILES_PER_PATCH >= 1) {
        patch0 = tile / (C::TILES_PER_PATCH > 0 ? C::TILES_PER_PATCH : 1);
        y0 = (tile - patch0 * C::TILES_PER_PATCH) * C::ROWS_PER_TILE;
      } else {
        patch0 = tile * PPT;
        y0 = 0;
      }
      int ky = 0, kx = 0, cc = 0;
#pragma unroll 1
      for (int s = 0; s < C::SPT; ++s) {
        mbar_wait(empty_bar(stage), phase ^ 1u);
        if (elect_one()) {
          const uint32_t lead_full = mapa_cluster(full_bar(stage), 0);
          const uint32_t a_dst = ring_base + stage * C::STAGE_BYTES;
          mbar_arrive_expect_tx_cluster(lead_full, C::STAGE_BYTES);
          if (ROWSHIFT) {
            tma_load_4d_pair(a_dst, &p.tmA[0], lead_full, (kx - 1) * 8, patch0, y0 - 1, cc * C::NPL);
          } else if (STRIDE == 1) {
            tma_load_4d_pair(a_dst, &p.tmA[0], lead_full, (kx - 1) * 8, y0 + ky - 1, patch0, cc * C::NPL);
          } else {
            const int xpar = (kx != 1), ypar = (ky != 1);
            tma_load_4d_pair(a_dst, &p.tmA[ypar * 2 + xpar], lead_full, (kx == 0) ? -8 : 0, y0 + ((ky == 0) ? -1 : 0), patch0,
                             cc * C::NPL);
          }
        }
        if (++cc == C::CIN_CHUNKS) {
          cc = 0;
          if (++kx == 3) { kx = 0; ++ky; }
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // ============================== UMMA issuer (leader CTA only, warp-uniform) ==============================
    if (rank == 0) {
      const uint32_t idesc = make_idesc_f16(2 * kTileM, N, p.act_bf16);
      constexpr uint32_t A_HI = noswizzle_desc_hi(128);
      constexpr uint32_t B_HI = kmajor_desc_hi(C::KCB);
      const uint32_t ring_a_lo = noswizzle_desc_lo(ring_base, C::PLANE_BYTES);
      const uint32_t w_lo = kmajor_desc_lo(w_base);
      mbar_wait(w_bar, 0);
      tc_fence_after();
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int grp = pair; grp < num_groups; grp += num_pairs, ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * N;
#pragma unroll
        for (int s = 0; s < C::SPT; ++s) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t a_lo = ring_a_lo + static_cast<uint32_t>(stage) * (C::STAGE_BYTES >> 4);
            if (ROWSHIFT) {
              const int kx = s / C::CIN_CHUNKS, cc = s - kx * C::CIN_CHUNKS;   // load unit = (kx, channel chunk)
#pragma unroll
              for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
                for (int k = 0; k < C::KCB / 32; ++k)
                  umma_f16_pair_w(d_tmem, a_lo + ((ky * C::ROW_BYTES + 2 * k * C::PLANE_BYTES) >> 4), A_HI,
                                  w_lo + ((((ky * 3 + kx) * C::CIN_CHUNKS + cc) * C::BH_BYTES) >> 4) + 2 * k, B_HI, idesc,
                                  (s | ky | k) != 0);
              }
            } else {
#pragma unroll
              for (int k = 0; k < C::KCB / 32; ++k)
                umma_f16_pair_w(d_tmem, a_lo + ((2 * k * C::PLANE_BYTES) >> 4), A_HI, w_lo + ((s * C::BH_BYTES) >> 4) + 2 * k,
                                B_HI, idesc, (s | k) != 0);
            }
            umma_commit_pair(empty_bar(stage));                        // frees the slot in both CTAs
            if (s == C::SPT - 1) umma_commit_pair(tfull_bar(acc));     // both CTAs' accumulators are complete
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else {
    // ============================== epilogue (both CTAs, each its own tile) ==============================
    const int q = warp & 3;  // TMEM lane quarter this warp may touch
    const int row_in_tile = q * 32 + lane;
    const long long total_patches = p.total_rows / C::PIX;
    int it = 0;
    for (int grp = pair; grp < num_groups; grp += num_pairs, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
      const int tile = grp * 2 + static_cast<int>(rank);
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * N;
      long long patch;
      int pix;
      if (ROWSHIFT && PPT > 1) {   // rows ordered (y, patch, x)
        patch = static_cast<long long>(tile) * PPT + (row_in_tile / HOUT) % PPT;
        pix = (row_in_tile / (HOUT * PPT)) * HOUT + row_in_tile % HOUT;
      } else {                     // rows ordered (patch, y, x)
        const long long row = static_cast<long long>(tile) * kTileM + row_in_tile;
        patch = row / C::PIX;
        pix = static_cast<int>(row - patch * C::PIX);
      }
      const bool valid = patch < total_patches;
      const int slot = planar_pixel_slot<HOUT, OUT_PARITY>(pix / HOUT, pix % HOUT);
      uint4* dst = reinterpret_cast<uint4*>(static_cast<uint16_t*>(p.out) + patch * (static_cast<long long>(N) * C::PIX)) + slot;
#pragma unroll
      for (int c0 = 0; c0 < N; c0 += 32) {
        uint32_t r[32];
        tmem_ld32(t_row + c0, r);
        tmem_ld_wait();
        uint32_t o[16];
#pragma unroll
        for (int j = 0; j < 16; ++j)
          o[j] = pack16_relu(__uint_as_float(r[2 * j]) + p.bias_v[c0 + 2 * j], __uint_as_float(r[2 * j + 1]) + p.bias_v[c0 + 2 * j + 1],
                             p.act_bf16);
        if (valid) {
#pragma unroll
          for (int j = 0; j < 4; ++j) dst[(c0 / 8 + j) * C::PIX] = make_uint4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(mapa_cluster(tempty_bar(acc), 0));
    }
  }

  // nobody leaves (and frees shared / tensor memory) while the peer may still read it or signal its barriers
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, C::TMEM_COLS);
  }
}

}  // namespace hn
