// conv3 + conv4 of the HardNet stack in ONE kernel (features[6..11], reference hardnet/HardNet.py:287-292):
//   3x3 stride-2 conv 32 -> 64 + BN + ReLU  ->  3x3 conv 64 -> 64 + BN + ReLU,
// with the 32 KB/patch activation between them resident in shared memory (never written to HBM: the two layers as
// separate kernels move 96 + 64 KB per patch, this kernel 64 + 32 KB).
//
// Work split: a CTA pair (tcgen05.mma.cta_group::2, M = 256) works on TWO patches at a time, one per CTA. A 16 x 16
// output map is two 128-pixel tiles (image rows 0-7 / 8-15); an MMA covers tile t of both CTAs' patches. Each CTA keeps
// half of the weight rows of BOTH layers resident, as in conv3x3_pair_kernel.
//
// conv3 (stride 2) reads the parity-planar conv2 output through TMA: one 9 KB box per (row parity, kx) - rows y0-1 .. y0+7
// of a parity sub-plane, shifted by the kx column offset; the ky taps of that parity are descriptor offsets of whole image
// rows (6 loads per tile). conv3's epilogue (bias + ReLU + 16-bit pack) does not store to global memory: it writes the
// activation into shared memory in the channel-planar layout = UMMA no-swizzle K-major operand, [plane][row -1..16][16 px][8 ch]
// (the halo rows are zeroed once and never written = the conv's zero padding in y).
//
// conv4's kx taps are STACKED ON N: the three kx taps share ONE read of the activation. Per ky the weights are a
// [192 = kx * 64 + c_out][64] tile, an MMA has N = 192 (96 clk of math for 4 KB of A; with one N = 64 MMA per tap the kernel
// was bound by the shared-memory pipe), and the conv is finished behind the MMAs:  out[y][x] = D0[y][x - 1] + D1[y][x] + D2[y][x + 1].
// An accumulator lane is a pixel and a 32-lane quarter is two image rows, so D2 is moved one lane down inside tensor memory
// (tcgen05.shift, a dedicated warp, once the tile's MMAs have retired) and D0 one lane up by warp shuffles in the epilogue;
// the row ends are masked = the conv's zero padding in x.
// Shared memory holds the activation double-buffered by patch (the conv3 epilogue of group i + 1 never waits for conv4 of
// group i) and a TMA ring of 11 boxes. Tensor memory: conv3 2 tiles x 64 columns (a tile's buffer is handed back as soon as
// the epilogue has read it) + conv4 2 tiles x 192 = 512.
//
// Issue order per group i of two patches:  conv3(i + 1) tile 0,  conv4(i) tile 0,  conv3(i + 1) tile 1,  conv4(i) tile 1
// (the TMA ring drains in bursts of 6 of its 11 boxes).
// Warps (20): 0 and 3 TMA producers (tile 0 / tile 1 boxes), 1 issuer / TMEM owner, 2 shifter, 4..19 epilogue: (tile, lane
// quarter, 32-channel half) each.
#pragma once

#include "common.cuh"
#include "tc_conv.cuh"
#include "tc_conv_pair.cuh"

#include <type_traits>
#include <utility>

namespace hn {

template <int N, class F, int... I>
__device__ __forceinline__ void static_for_impl(F&& f, std::integer_sequence<int, I...>) {
  (f(std::integral_constant<int, I>{}), ...);
}
// f(integral_constant<int, 0>) ... f(integral_constant<int, N - 1>): a compile-time unrolled loop whose index is a constant
template <int N, class F>
__device__ __forceinline__ void static_for(F&& f) {
  static_for_impl<N>(static_cast<F&&>(f), std::make_integer_sequence<int, N>{});
}

#ifdef HN_C34_TRACE
// Diagnostic build only (-DHN_C34_TRACE): cycles the roles of CTA 0 spend blocked on each barrier, summed over a launch.
static __device__ unsigned long long hn_c34_trace[16];
#define C34_WAIT(slot, bar, par) do { const long long t0__ = clock64(); mbar_wait(bar, par); \
  if (blockIdx.x == 0 && lane == 0) atomicAdd(&hn_c34_trace[slot], static_cast<unsigned long long>(clock64() - t0__)); } while (0)
#define C34_T0() const long long ts__ = clock64()
#define C34_ACC(slot) do { if (blockIdx.x == 0 && lane == 0) atomicAdd(&hn_c34_trace[slot], static_cast<unsigned long long>(clock64() - ts__)); } while (0)
#else
#define C34_WAIT(slot, bar, par) mbar_wait(bar, par)
#define C34_T0() do { } while (0)
#define C34_ACC(slot) do { } while (0)
#endif

constexpr int kC34SThreads = 20 * 32;

__device__ __forceinline__ void tmem_ld16_c34(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

struct C34SCfg {
  static constexpr int UNITS = 6, ROWS = 9;
  static constexpr uint32_t A3_PLANE = ROWS * 256;
  static constexpr uint32_t A3_BYTES = 4 * A3_PLANE;
  static constexpr int STAGES = 11;
  static constexpr uint32_t W3_BLK = 32 * 64;
  static constexpr uint32_t W3_BYTES = 9 * W3_BLK;
  static constexpr uint32_t W4_KY = 96 * 128;           // this CTA's 96 of the 192 stacked rows of one ky, 64 input channels
  static constexpr uint32_t W4_BYTES = 3 * W4_KY;
  static constexpr uint32_t MID_PLANE = 18 * 256;       // image rows -1 .. 16
  static constexpr uint32_t MID_BUF = 8 * MID_PLANE;    // 64 channels
  static constexpr uint32_t MID_BYTES = 2 * MID_BUF;
  static constexpr size_t SMEM = size_t(W3_BYTES) + W4_BYTES + MID_BYTES + size_t(STAGES) * A3_BYTES + 1024 + 320;   // 34 barriers + TMEM slot
  static_assert(SMEM <= 227 * 1024, "shared memory budget");
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kC34SThreads, 1)
conv34_stack_kernel(const __grid_constant__ Conv34Params p) {
  using C = C34SCfg;
  constexpr int STAGES = C::STAGES;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;   // identical in both CTAs
  const uint32_t w3_base = base;
  const uint32_t w4_base = w3_base + C::W3_BYTES;
  const uint32_t mid_base = w4_base + C::W4_BYTES;
  const uint32_t ring_base = mid_base + C::MID_BYTES;
  const uint32_t bar_base = ring_base + STAGES * C::A3_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto t3full_bar = [&](int t) { return bar_base + 8u * (2 * STAGES + t); };
  auto t3empty_bar = [&](int t) { return bar_base + 8u * (2 * STAGES + 2 + t); };
  auto t4full_bar = [&](int t) { return bar_base + 8u * (2 * STAGES + 4 + t); };
  auto t4empty_bar = [&](int t) { return bar_base + 8u * (2 * STAGES + 6 + t); };
  auto mma4_bar = [&](int t) { return bar_base + 8u * (2 * STAGES + 8 + t); };
  const uint32_t mid_bar = bar_base + 8u * (2 * STAGES + 10);
  const uint32_t w_bar = bar_base + 8u * (2 * STAGES + 11);
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 12);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw_addr));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pr = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
  const int num_groups = (p.n_patches + 1) / 2;                    // a group = two consecutive patches, one per CTA
  const int n_it = pr < num_groups ? (num_groups - pr + num_pairs - 1) / num_pairs : 0;  // groups of this pair

#ifdef HN_C34_TRACE
  const long long c34_start = clock64();
#endif
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmA[0]);
    tma_prefetch_desc(&p.tmA[1]);
    tma_prefetch_desc(&p.tmA[2]);
    tma_prefetch_desc(&p.tmA[3]);
    tma_prefetch_desc(&p.tmB3);
    tma_prefetch_desc(&p.tmB4);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < STAGES; ++s) {
        mbar_init(full_bar(s), 2);    // one arrive.expect_tx per CTA of the pair (leader's copy)
        mbar_init(empty_bar(s), 1);   // multicast tcgen05.commit
      }
      for (int t = 0; t < 2; ++t) {
        mbar_init(t3full_bar(t), 1);     // multicast tcgen05.commit
        mbar_init(t3empty_bar(t), 16);   // the tile's eight epilogue warps of each CTA (leader's copy)
        mbar_init(mma4_bar(t), 1);       // conv4 MMAs of the tile retired -> shifter
        mbar_init(t4full_bar(t), 1);     // multicast tcgen05.commit behind the shifts
        mbar_init(t4empty_bar(t), 16);
      }
      mbar_init(mid_bar, 32);            // sixteen epilogue warps of each CTA (leader's copy)
      mbar_init(w_bar, 2);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc_pair(tmem_slot, 512);
    tmem_relinquish_pair();
  }
  // zero both activation buffers once: the halo rows (-1 and 16) are never written = the conv's zero padding
  {
    uint4* mid = reinterpret_cast<uint4*>(smem_raw + (mid_base - raw_addr));
    for (uint32_t i = threadIdx.x; i < C::MID_BYTES / 16; i += kC34SThreads) mid[i] = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // the peer's barriers are initialised and its TMEM is allocated before anyone signals it
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0 || warp == 3) {
    // ============================== TMA producers (both CTAs, warp-uniform) ==============================
    // Warp 0 loads the boxes of tile 0, warp 3 those of tile 1 (a cp.async.bulk.tensor issue blocks its thread until the TMA
    // unit has taken the request; two threads keep two requests in flight). Ring slots are dealt in load order.
    const int pw = warp == 0 ? 0 : 1;
    if (pw == 0) {
      const uint32_t lead_w_bar = mapa_cluster(w_bar, 0);
      if (elect_one()) {
        mbar_arrive_expect_tx_cluster(lead_w_bar, C::W3_BYTES + C::W4_BYTES);
#pragma unroll 1
        for (int kb = 0; kb < 9; ++kb) tma_load_2d_pair(w3_base + kb * C::W3_BLK, &p.tmB3, lead_w_bar, kb * 32, static_cast<int>(rank) * 32);
        // stacked conv4 weights: row n = kx * 64 + c_out of the [192][64] tile of one ky; this CTA holds rows 96 * rank .. + 95
        // as three 32-row boxes of the [64][9 * 64] weight matrix
#pragma unroll 1
        for (int kyg = 0; kyg < 9; ++kyg) {
          const int ky = kyg / 3, g = kyg - 3 * ky;
          const int n0 = 96 * static_cast<int>(rank) + 32 * g;
          tma_load_2d_pair(w4_base + ky * C::W4_KY + g * 4096, &p.tmB4, lead_w_bar, (ky * 3 + (n0 >> 6)) * 64, n0 & 63);
        }
      }
      __syncwarp();
    }
    int stage = pw * C::UNITS;
    uint32_t phase = 0;
    for (int it = 0; it < n_it; ++it) {
      // a patch index past the batch reads stale or out-of-range (zero-filled) data; its results are never stored
      const int patch = 2 * (pr + it * num_pairs) + static_cast<int>(rank);
#pragma unroll 1
      for (int u = 0; u < C::UNITS; ++u) {
        C34_WAIT(9, empty_bar(stage), phase ^ 1u);
        C34_T0();
        if (elect_one()) {
          const uint32_t lead_full = mapa_cluster(full_bar(stage), 0);
          mbar_arrive_expect_tx_cluster(lead_full, C::A3_BYTES);
          // u = yp * 3 + kx: yp 0 = odd input rows (taps ky 0 and 2), yp 1 = even input rows (tap ky 1);
          // input x = 2*ox + kx - 1: kx=0 -> odd column ox-1, kx=1 -> even column ox, kx=2 -> odd column ox
          const int yp = u / 3, kx = u - yp * 3;
          const int xpar = (kx != 1), ypar = (yp == 0);
          tma_load_4d_pair(ring_base + stage * C::A3_BYTES, &p.tmA[ypar * 2 + xpar], lead_full, (kx == 0) ? -8 : 0, 8 * pw - 1, patch, 0);
        }
        __syncwarp();
        if (pw == 0) C34_ACC(12);
        if (++stage >= STAGES) { stage -= STAGES; phase ^= 1u; }
      }
      // skip the other producer's six slots
      stage += C::UNITS;
      if (stage >= STAGES) { stage -= STAGES; phase ^= 1u; }
    }
  } else if (warp == 1) {
    // ============================== UMMA issuer (leader CTA only, warp-uniform) ==============================
    if (rank == 0) {
      const uint32_t idesc3 = make_idesc_f16(2 * kTileM, 64, p.act_bf16);
      const uint32_t idesc4 = make_idesc_f16(2 * kTileM, 192, p.act_bf16);
      constexpr uint32_t A_HI = noswizzle_desc_hi(128);
      constexpr uint32_t B3_HI = kmajor_desc_hi(64);
      constexpr uint32_t B4_HI = kmajor_desc_hi(128);
      const uint32_t ring_a_lo = noswizzle_desc_lo(ring_base, C::A3_PLANE);
      const uint32_t mid_a_lo = noswizzle_desc_lo(mid_base, C::MID_PLANE);
      const uint32_t w3_lo = kmajor_desc_lo(w3_base);
      const uint32_t w4_lo = kmajor_desc_lo(w4_base);
      mbar_wait(w_bar, 0);
      tc_fence_after();
      int stage = 0;
      uint32_t phase = 0;
      // A satisfied mbarrier.try_wait still costs the polling warp > 100 clk of latency and a conv3 load unit is only 2 - 4 MMAs
      // (96 - 192 clk of tensor-pipe work): the barrier of the NEXT unit is probed before the MMAs of the current one are issued,
      // so that latency overlaps the issue; only a box that really has not landed yet is waited for.
      uint32_t ready = 0;
      auto conv3_unit = [&](auto t_c, auto u_c) {
        constexpr int t = decltype(t_c)::value, u = decltype(u_c)::value;
        const uint32_t d_tmem = tmem_base + t * 64;
        if (!ready) C34_WAIT(0, full_bar(stage), phase);
        {
          const int ns = stage + 1 == STAGES ? 0 : stage + 1;
          ready = mbar_try_wait(full_bar(ns), ns == 0 ? phase ^ 1u : phase);
        }
        if (elect_one()) {
          const uint32_t a_lo = ring_a_lo + static_cast<uint32_t>(stage) * (C::A3_BYTES >> 4);
          constexpr int yp = u / 3, kx = u - yp * 3;
          if constexpr (yp == 0) {
#pragma unroll
            for (int kyi = 0; kyi < 2; ++kyi) {   // ky = 0 (rows y0-1 ..) and ky = 2 (rows y0 ..)
              const int ky = 2 * kyi;
#pragma unroll
              for (int k = 0; k < 2; ++k)
                umma_f16_pair_w(d_tmem, a_lo + ((kyi * 256 + 2 * k * C::A3_PLANE) >> 4), A_HI,
                                w3_lo + (((ky * 3 + kx) * C::W3_BLK) >> 4) + 2 * k, B3_HI, idesc3, (u | kyi | k) != 0);
            }
          } else {
#pragma unroll
            for (int k = 0; k < 2; ++k)
              umma_f16_pair_w(d_tmem, a_lo + ((256 + 2 * k * C::A3_PLANE) >> 4), A_HI, w3_lo + (((3 + kx) * C::W3_BLK) >> 4) + 2 * k,
                              B3_HI, idesc3, 1u);
          }
          umma_commit_pair(empty_bar(stage));
          if (u == C::UNITS - 1) umma_commit_pair(t3full_bar(t));
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      };
      for (int j = -1; j < n_it; ++j) {
        static_for<2>([&](auto t_c) {
          constexpr int t = decltype(t_c)::value;
          if (j + 1 < n_it) {
            if (j >= 0) {   // the conv3 epilogue of group j has read this tile's accumulator
              C34_WAIT(2, t3empty_bar(t), j & 1);
              tc_fence_after();
            }
            static_for<C::UNITS>([&](auto u_c) { conv3_unit(t_c, u_c); });
          }
          if (j >= 0) {
            if (t == 0) C34_WAIT(1, mid_bar, j & 1);   // the conv3 epilogue of group j has written its activation buffer (both CTAs)
            if (j >= 1) C34_WAIT(10, t4empty_bar(t), (j - 1) & 1);   // the conv4 epilogue of group j - 1 has drained this accumulator
            tc_fence_after();
            if (elect_one()) {
              const uint32_t a_buf = mid_a_lo + (((j & 1) * C::MID_BUF) >> 4);
              const uint32_t d_tmem = tmem_base + 128 + t * 192;
#pragma unroll
              for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  umma_f16_pair_w(d_tmem, a_buf + (((8 * t + ky) * 256 + 2 * k * C::MID_PLANE) >> 4), A_HI,
                                  w4_lo + ((ky * C::W4_KY) >> 4) + 2 * k, B4_HI, idesc4, (ky | k) != 0);
              }
              umma_commit_pair(mma4_bar(t));
            }
            __syncwarp();
          }
        });
      }
    }
  } else if (warp == 2) {
    // ============================== shifter (leader CTA only) ==============================
    // D2 (columns 128..191 of a conv4 accumulator) is needed one pixel to the left: tcgen05.shift moves the rows of every
    // 32-lane quarter down by one lane, 8 columns per instruction, in both CTAs' tensor memory (lanes 15 and 31 = x 15 receive
    // a value that the epilogue masks). The shift is not ordered behind earlier MMAs by itself: it waits for the tile's
    // mma4 barrier; the commit behind it publishes the accumulator to the epilogue warps of both CTAs.
    if (rank == 0) {
      for (int it = 0; it < n_it; ++it) {
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          C34_WAIT(11, mma4_bar(t), it & 1);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t ds = tmem_base + 128 + t * 192 + 128;
#pragma unroll
            for (int c8 = 0; c8 < 8; ++c8) asm volatile("tcgen05.shift.cta_group::2.down [%0];" ::"r"(ds + c8 * 8) : "memory");
            umma_commit_pair(t4full_bar(t));
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ============================== epilogue (both CTAs, each its own patch) ==============================
    const int e = warp - 4;
    const int q = warp & 3;         // TMEM lane quarter this warp may touch
    const int t = (e >> 2) >> 1;    // tile (image rows 8t .. 8t + 7)
    const int h = (e >> 2) & 1;     // channels 32h .. 32h + 31
    const int y = 8 * t + 2 * q + (lane >> 4), x = lane & 15;
    const uint32_t lead_mid_bar = mapa_cluster(mid_bar, 0);
    const uint32_t lead_t3empty = mapa_cluster(t3empty_bar(t), 0);
    const uint32_t lead_t4empty = mapa_cluster(t4empty_bar(t), 0);
    uint8_t* mid_px = smem_raw + (mid_base - raw_addr) + (4 * h) * C::MID_PLANE + (y + 1) * 256 + x * 16;   // buffer 0, first plane of this half
    const int out_slot = planar_pixel_slot<16, true>(y, x);
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const float m_left = x > 0 ? 1.f : 0.f, m_right = x < 15 ? 1.f : 0.f;

    auto epilogue4 = [&](int it) {
      if (e == 0) C34_WAIT(6, t4full_bar(t), it & 1);
      mbar_wait(t4full_bar(t), it & 1);
      tc_fence_after();
      const long long patch = 2ll * (pr + it * num_pairs) + rank;
      const bool valid = patch < p.n_patches;
      const uint32_t t_row = t_lane + 128 + t * 192 + 32 * h;
      uint4* dst = reinterpret_cast<uint4*>(static_cast<uint16_t*>(p.out) + patch * (64ll * 256)) + (4 * h) * 256 + out_slot;
#pragma unroll
      for (int c0 = 0; c0 < 32; c0 += 16) {
        uint32_t r0[16], r1[16], r2[16];
        tmem_ld16_c34(t_row + c0, r0);          // kx = 0: this lane holds the contribution to the pixel on its right
        tmem_ld16_c34(t_row + 64 + c0, r1);     // kx = 1
        tmem_ld16_c34(t_row + 128 + c0, r2);    // kx = 2, already moved one lane down: the contribution of pixel x + 1
        tmem_ld_wait();
        if (c0 == 16) {   // everything this warp needs of the accumulator is in registers: hand it back before the arithmetic
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(lead_t4empty);
        }
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float from_left = __shfl_up_sync(0xffffffffu, __uint_as_float(r0[j]), 1);
          v[j] = fmaf(__uint_as_float(r2[j]), m_right, fmaf(from_left, m_left, __uint_as_float(r1[j]) + p.bias4[32 * h + c0 + j]));
        }
        if (valid) {
#pragma unroll
          for (int j = 0; j < 2; ++j)
            dst[(c0 / 8 + j) * 256] = make_uint4(pack16_relu(v[8 * j], v[8 * j + 1], p.act_bf16), pack16_relu(v[8 * j + 2], v[8 * j + 3], p.act_bf16),
                                                 pack16_relu(v[8 * j + 4], v[8 * j + 5], p.act_bf16), pack16_relu(v[8 * j + 6], v[8 * j + 7], p.act_bf16));
        }
      }
    };

    for (int it = 0; it < n_it; ++it) {
      if (e == 0) C34_WAIT(5, t3full_bar(t), it & 1);
      mbar_wait(t3full_bar(t), it & 1);   // conv3 accumulator of this tile, group `it`
      tc_fence_after();
      C34_T0();
      {
        uint32_t r[32];
        tmem_ld32(t_lane + t * 64 + 32 * h, r);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(lead_t3empty);   // conv3 of the next group may overwrite the accumulator
        // this buffer's previous reader, conv4 of group it - 2, retired before conv3 of group `it` did (issue order)
        uint8_t* d = mid_px + (it & 1) * C::MID_BUF;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t o[4];
#pragma unroll
          for (int i = 0; i < 4; ++i)
            o[i] = pack16_relu(__uint_as_float(r[8 * j + 2 * i]) + p.bias3[32 * h + 8 * j + 2 * i],
                               __uint_as_float(r[8 * j + 2 * i + 1]) + p.bias3[32 * h + 8 * j + 2 * i + 1], p.act_bf16);
          *reinterpret_cast<uint4*>(d + j * C::MID_PLANE) = make_uint4(o[0], o[1], o[2], o[3]);
        }
      }
      fence_proxy_async_smem();   // generic-proxy writes -> visible to the tensor cores (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(lead_mid_bar);
      if (e == 0) C34_ACC(7);
      if (it > 0) epilogue4(it - 1);
      if (e == 0) C34_ACC(8);
    }
    if (n_it > 0) epilogue4(n_it - 1);
  }

  // nobody leaves (and frees shared / tensor memory) while the peer may still read it or signal its barriers
  tc_fence_before();
  __syncthreads();
#ifdef HN_C34_TRACE
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    atomicAdd(&hn_c34_trace[3], static_cast<unsigned long long>(clock64() - c34_start));
    atomicAdd(&hn_c34_trace[4], static_cast<unsigned long long>(n_it));
  }
#endif
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, 512);
  }
}

}  // namespace hn
