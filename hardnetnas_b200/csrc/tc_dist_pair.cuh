// CTA-pair (tcgen05.mma.cta_group::2, M = 256) version of the SHORTLIST matching GEMM of tc_dist.cuh
// (FDLNet-master/utils/eval_utils.py:113-114,168-175 behind hn_match). Each CTA of a pair keeps 256 query rows resident
// (two 128-row M-blocks, K = 128) and loads HALF of every 128-row gallery tile (64 rows); one MMA covers an M-block of
// both CTAs against the whole tile. Per SM an MMA step then reads A (32 wavefronts) + half of B (16) instead of 64,
// which takes the N = 128 GEMM off the shared-memory port limit, and the gallery streams through each SM's L2 port once
// per 512 query rows instead of once per 256. The epilogue (top-4 chunks per row + their maxima) and the output format
// are those of dist_kernel<2, EPI_SHORTLIST>; the signalling protocol is the one of tc_conv_pair.cuh.
// F8: e4m3 operand rows (see tc_dist.cuh): an A block is one 128-byte K block instead of two and a stage is one 8 KB half-tile
// instead of two k-blocks, with kind::f8f6f4 MMAs (umma_f8_pair_w). The stage count stays kMpStages: the same number of
// gallery tiles in flight, in half the shared memory.
#pragma once

#include "tc_conv_pair.cuh"
#include "tc_dist.cuh"

namespace hn {

constexpr int kMpStages = 6;                       // gallery half-tiles (both k-blocks, 16 KB; F8: 8 KB) in flight per CTA
constexpr uint32_t kMpABlk = kDistTile * 128;      // one 128-row x 64-element A block (F8: 128 e4m3)
constexpr uint32_t kMpBBlk = 64 * 128;             // this CTA's 64-row x 64-element half of a B k-block (F8: 128 e4m3)
template <bool F8>
constexpr int mp_k_blocks() { return F8 ? 1 : 2; }
template <bool F8>
constexpr uint32_t mp_stage_bytes() { return mp_k_blocks<F8>() * kMpBBlk; }   // all k-blocks of a half tile
template <bool F8>
constexpr size_t mp_smem_bytes() { return 2 * mp_k_blocks<F8>() * kMpABlk + kMpStages * mp_stage_bytes<F8>() + 1024 + 256; }
// The epilogue (per row: maxima of sixteen 8-column chunks per tile + a sorted insert) is the longest step per tile, so
// every 32-row lane quarter of an accumulator is shared by TWO warps, each reducing 64 of the 128 columns into its own
// top-kTopC list (the lists of the two halves are separate slots of the candidate table).
constexpr int kMpEpiWarps = 16;
constexpr int kMpThreads = 64 + kMpEpiWarps * 32;

template <bool F8>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kMpThreads, 1) match_pair_kernel(const __grid_constant__ DistParams p) {
  constexpr int MB = 2;
  constexpr int KB = mp_k_blocks<F8>();
  constexpr uint32_t kMpStage = mp_stage_bytes<F8>();
  const DistSide& sd = p.side[0];
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  const uint32_t a_base = base;                              // [mb][kb] blocks
  const uint32_t b_base = base + MB * KB * kMpABlk;
  const uint32_t bar_base = b_base + kMpStages * kMpStage;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kMpStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * kMpStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * kMpStages + 2 + a); };
  const uint32_t afull_bar = bar_base + 8u * (2 * kMpStages + 4);
  const uint32_t aempty_bar = bar_base + 8u * (2 * kMpStages + 5);
  const uint32_t tmem_slot = bar_base + 8u * (2 * kMpStages + 6);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw_addr));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;

  const int m_blocks = static_cast<int>((sd.Na + 2 * MB * kDistTile - 1) / (2 * MB * kDistTile));   // 512 query rows per pair
  const int n_tiles = static_cast<int>((sd.Nb + kDistTile - 1) / kDistTile);
  const int num_items = m_blocks * p.segments;
  auto seg_range = [&](int seg, int& t0, int& t1) {
    t0 = static_cast<int>(static_cast<long long>(n_tiles) * seg / p.segments);
    t1 = static_cast<int>(static_cast<long long>(n_tiles) * (seg + 1) / p.segments);
  };

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&sd.tmA);
    tma_prefetch_desc(&sd.tmB);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < kMpStages; ++s) {
        mbar_init(full_bar(s), 2);     // one arrive.expect_tx per CTA (leader's copy is the live one)
        mbar_init(empty_bar(s), 1);    // multicast tcgen05.commit
      }
      for (int a = 0; a < 2; ++a) {
        mbar_init(tfull_bar(a), 1);    // multicast tcgen05.commit
        mbar_init(tempty_bar(a), 2 * kMpEpiWarps);  // the epilogue warps of both CTAs (leader's copy)
      }
      mbar_init(afull_bar, 2);
      mbar_init(aempty_bar, 1);        // multicast tcgen05.commit
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc_pair(tmem_slot, 512);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ============================== TMA producer (both CTAs, warp-uniform) ==============================
    const uint32_t lead_afull = mapa_cluster(afull_bar, 0);
    int stage = 0;
    uint32_t phase = 0, a_phase = 0;
    for (int item = pair; item < num_items; item += num_pairs) {
      const int mblk = item / p.segments, seg = item - mblk * p.segments;
      int t0, t1;
      seg_range(seg, t0, t1);
      mbar_wait(aempty_bar, a_phase ^ 1u);
      if (elect_one()) {
        mbar_arrive_expect_tx_cluster(lead_afull, MB * KB * kMpABlk);
        const int row0 = (mblk * 2 + static_cast<int>(rank)) * MB * kDistTile;
#pragma unroll
        for (int mb = 0; mb < MB; ++mb)
#pragma unroll
          for (int kb = 0; kb < KB; ++kb)
            tma_load_2d_pair(a_base + (mb * KB + kb) * kMpABlk, &sd.tmA, lead_afull, kb * 64, row0 + mb * kDistTile);
      }
      __syncwarp();
      a_phase ^= 1u;
      for (int t = t0; t < t1; ++t) {
        mbar_wait(empty_bar(stage), phase ^ 1u);
        if (elect_one()) {
          const uint32_t lead_full = mapa_cluster(full_bar(stage), 0);
          mbar_arrive_expect_tx_cluster(lead_full, kMpStage);
          const int grow = t * kDistTile + static_cast<int>(rank) * 64;
#pragma unroll
          for (int kb = 0; kb < KB; ++kb) tma_load_2d_pair(b_base + stage * kMpStage + kb * kMpBBlk, &sd.tmB, lead_full, kb * 64, grow);
        }
        __syncwarp();
        if (++stage == kMpStages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // ============================== UMMA issuer (leader CTA only) ==============================
    if (rank == 0) {
      const uint32_t idesc = make_idesc_f16(2 * kDistTile, kDistTile, 0);
      constexpr uint32_t HI = kmajor_desc_hi(128);
      const uint32_t a_lo0 = kmajor_desc_lo(a_base);
      const uint32_t b_lo0 = kmajor_desc_lo(b_base);
      int stage = 0;
      uint32_t phase = 0, a_phase = 0;
      int it = 0;
      for (int item = pair; item < num_items; item += num_pairs) {
        const int mblk = item / p.segments, seg = item - mblk * p.segments;
        int t0, t1;
        seg_range(seg, t0, t1);
        mbar_wait(afull_bar, a_phase);
        a_phase ^= 1u;
        tc_fence_after();
        for (int t = t0; t < t1; ++t, ++it) {
          const int acc = it & 1;
          const uint32_t acc_phase = (it >> 1) & 1;
          mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t b_lo = b_lo0 + static_cast<uint32_t>(stage) * (kMpStage >> 4);
#pragma unroll
            for (int mb = 0; mb < MB; ++mb) {
              const uint32_t d_tmem = tmem_base + (acc * MB + mb) * kDistTile;
#pragma unroll
              for (int kb = 0; kb < KB; ++kb) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const uint32_t a_lo = a_lo0 + (((mb * KB + kb) * kMpABlk) >> 4) + 2u * k, b_lo_k = b_lo + ((kb * kMpBBlk) >> 4) + 2u * k;
                  if constexpr (F8) umma_f8_pair_w(d_tmem, a_lo, HI, b_lo_k, HI, idesc, (kb | k) != 0);
                  else umma_f16_pair_w(d_tmem, a_lo, HI, b_lo_k, HI, idesc, (kb | k) != 0);
                }
              }
            }
            umma_commit_pair(empty_bar(stage));
            umma_commit_pair(tfull_bar(acc));
          }
          __syncwarp();
          if (++stage == kMpStages) { stage = 0; phase ^= 1u; }
        }
        if (elect_one()) umma_commit_pair(aempty_bar);   // the resident query blocks of both CTAs may be overwritten
        __syncwarp();
      }
    }
  } else {
    // ============================== epilogue (both CTAs): top-kTopC chunks per row ==============================
    const int q = warp & 3;
    const int mb = (warp - 2) >> 3;          // M-block of this CTA
    const int half = ((warp - 2) >> 2) & 1;  // which 64 of the tile's 128 columns
    int it = 0;
    for (int item = pair; item < num_items; item += num_pairs) {
      const int mblk = item / p.segments, seg = item - mblk * p.segments;
      int t0, t1;
      seg_range(seg, t0, t1);
      const long long row = static_cast<long long>((mblk * 2 + static_cast<int>(rank)) * MB + mb) * kDistTile + q * 32 + lane;
      const bool row_ok = row < sd.Na;
      float tb[kTopC];
      int tc[kTopC];
#pragma unroll
      for (int i = 0; i < kTopC; ++i) { tb[i] = -__int_as_float(0x7f800000); tc[i] = 0; }
      const uint32_t lead_tempty0 = mapa_cluster(tempty_bar(0), 0), lead_tempty1 = mapa_cluster(tempty_bar(1), 0);
      for (int t = t0; t < t1; ++t, ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        const long long col0 = static_cast<long long>(t) * kDistTile + half * 64;
        mbar_wait(tfull_bar(acc), acc_phase);
        tc_fence_after();
        const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + (acc * MB + mb) * kDistTile + half * 64;
        const bool ragged = col0 + 64 > sd.Nb;
        uint32_t r[2][32];
#pragma unroll
        for (int gq = 0; gq < 2; ++gq) tmem_ld32(t_row + gq * 32, r[gq]);
        tmem_ld_wait();
        float cm[8];   // this row's maxima of the eight chunks of this 64-column half
#pragma unroll
        for (int gq = 0; gq < 2; ++gq) {
          const int c0 = gq * 32;
          float v[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[gq][j]);
          if (ragged) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (col0 + c0 + j >= sd.Nb) v[j] = -__int_as_float(0x7f800000);
          }
#pragma unroll
          for (int s = 0; s < 32 / kChunk; ++s) {
            const float* w = v + s * kChunk;
            const float m = fmaxf(max3(w[0], w[1], w[2]), max3(max3(w[3], w[4], w[5]), w[6], w[7]));
            cm[gq * 4 + s] = m;
            if (m > tb[kTopC - 1]) {
              const int id = static_cast<int>((col0 + c0) / kChunk) + s;
              const bool g0 = m > tb[0], g1 = m > tb[1], g2 = m > tb[2];
              tb[3] = g2 ? tb[2] : m;               tc[3] = g2 ? tc[2] : id;
              tb[2] = g2 ? (g1 ? tb[1] : m) : tb[2]; tc[2] = g2 ? (g1 ? tc[1] : id) : tc[2];
              tb[1] = g1 ? (g0 ? tb[0] : m) : tb[1]; tc[1] = g1 ? (g0 ? tc[0] : id) : tc[1];
              tb[0] = g0 ? m : tb[0];               tc[0] = g0 ? id : tc[0];
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(acc ? lead_tempty1 : lead_tempty0);
        if (sd.block_max != nullptr) {   // warp-uniform: column side of mutual NN (hn_match_mutual)
          const float bm = warp_chunk_max8(cm, lane);
          const long long cb = col0 / kChunk + (lane >> 2);
          const long long rb = row >> 5;
          if ((lane & 3) == 0 && cb * kChunk < sd.Nb && rb < sd.n_row_blocks) sd.block_max[cb * sd.n_row_blocks + rb] = bm;
        }
      }
      if (row_ok) store_cand_list(sd.cand, sd.cand_val, (row * p.segments + seg) * 2 + half, tb, tc);
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, 512);
  }
}

}  // namespace hn
