// Fused front of the HardNet stack: input_norm + conv 1->32 + BN + ReLU (features[0..2]) and conv 32->32 + BN + ReLU
// (features[3..5], reference hardnet/HardNet.py:281-286,306-310) in ONE persistent kernel. The 64 KB/patch stage-1
// activation never leaves the SM: its epilogue writes it to shared memory in a channel-planar, row-haloed layout
//     act1[plane = c / 8][slot = (y + 1) * 32 + x][c % 8]            (fp16/bf16, 16 B per slot, 34 x 32 slots per plane)
// which IS a UMMA no-swizzle K-major operand (8 consecutive slots x 16 B = one core matrix, SBO = 128 B,
// LBO = plane pitch), so a ky tap of conv2 is the same buffer viewed 32 slots further on - no im2col copy.
//
// conv2 runs with the three kx taps STACKED ON N:  D'[p, kx * 32 + co] = sum_{ky, ci} act1[p + (ky - 1) row, ci] *
// w[ky, kx, ci, co]  (M = 128 pixels = 4 image rows, N = 96, K = 3 x 32), so each A tile is read from shared memory
// 3 times instead of 9 (SS-mode UMMA is bound by the 128 B/clk shared-memory port when N is small). The epilogue
// finishes the conv:  out[y, x] = D'0[y, x - 1] + D'1[y, x] + D'2[y, x + 1]. A TMEM lane quarter is exactly one image row,
// so D'2 is moved one lane down with tcgen05.shift (in tensor memory, behind the MMAs), D'0 one lane up with half a
// shuffle per value (fp16 pairs), and the edge lanes are masked = the conv's zero padding in x.
//
// The stage-1 BatchNorm shift rides in the spare K slots of the stage-1 GEMM (K = 9 taps padded to 16): im2col columns 9
// and 10 are the constant 1 and the matching weight rows hold the shift split into a 16-bit hi + lo pair, so the tensor
// core adds it in fp32 and the stage-1 epilogue is just TMEM -> ReLU/pack (one F2FP per two values) -> shared memory.
//
// Warps (20): 0-3 stage-1 epilogue (TMEM -> act1 in smem), 4-11 conv2 epilogue (two groups of four, one per
// accumulator pair), 12 TMEM owner + UMMA issuer A (stage 1 + even conv2 tiles), 13-16 loaders (normalise + im2col of
// the 1-channel input), 17 UMMA issuer B (odd conv2 tiles), 18-19 shifters (tcgen05.shift of the even / odd tiles).
// Why several issuing warps: an mbarrier.try_wait costs the polling warp ~180 cycles even when the barrier is already
// complete (tools/issue_probe.cu), and one conv2 tile is only 336 cycles of tensor-pipe work. A single warp that polls
// accumulator-free, issues, polls MMAs-retired and shifts leaves the pipe idle between tiles; with the tiles dealt to
// two issuers and the shifts to two more warps those latencies overlap each other and the MMAs.
#pragma once

#include "clip.cuh"
#include "common.cuh"
#include "l1_tc.cuh"
#include "tc_conv.cuh"

namespace hn {

constexpr int kFfThreads = 20 * 32;
constexpr int kFfIssuer = 12;
constexpr int kFfLoader0 = 13;   // 4 loader warps: 13..16
constexpr int kFfIssuerB = 17;
constexpr int kFfShift0 = 18;    // 2 shifter warps: 18, 19
constexpr uint32_t kFfPlane = 34 * 32 * 16;   // one 8-channel plane of the haloed stage-1 output
constexpr uint32_t kFfAct1 = 4 * kFfPlane;    // 69 632 B per buffer
constexpr uint32_t kFfA1 = 8 * 4096;          // eight 128 x 16 im2col tiles of the input patch
constexpr uint32_t kFfW2Tap = 96 * 32 * 2;    // one ky: [kx * 32 + co][ci]
constexpr uint32_t kFfW2 = 3 * kFfW2Tap;      // 18 432 B
constexpr uint32_t kFfW1 = 1024;
constexpr int kFfRawDepth = 4;                 // raw input patches prefetched ahead of the loaders (bulk async copies)
constexpr uint32_t kFfRaw = kFfRawDepth * 4096;
constexpr uint32_t kFfStage = 8 * 2048;       // PW2 only: one 32-pixel x 32-channel output staging tile per epilogue warp
// FDW (PW2 + the block's stride-2 depthwise conv / max-pool in the same kernel): the pointwise output of a whole patch stays
// in shared memory (4 planes x 1024 pixels x 16 B, row/column parity sub-planes so the stride-2 taps of consecutive output
// columns are consecutive 16-byte slots) and only the 16 x 16 x 32 result (16 KB/patch instead of 64 KB) is written. The
// 64 KB tile takes the place of the second stage-1 buffer: stage 1 is single-buffered in this variant.
constexpr uint32_t kFfAct2 = 4 * 1024 * 16;
constexpr uint32_t kFfDwW = 26 * 32 * 2;      // fp16 depthwise weights [k * k <= 25][32] + bias [32]
constexpr size_t kFfSmem = kFfA1 + 2 * kFfAct1 + kFfW2 + kFfW1 + kFfRaw + kFfStage + 256 /*barriers*/ + 256 /*biases + reductions*/ + 1024 /*align*/;
static_assert(kFfSmem <= 227 * 1024, "smem budget");

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}

#ifdef HN_FF_TRACE
// Diagnostic build only (-DHN_FF_TRACE): cycles each role of CTA 0 spends blocked on each barrier, summed over the launch.
__device__ unsigned long long hn_ff_trace[32];
#define HN_FF_T0() const long long t0__ = clock64()
#define HN_FF_ACC(slot) do { if (blockIdx.x == 0 && lane == 0) atomicAdd(&hn_ff_trace[slot], static_cast<unsigned long long>(clock64() - t0__)); } while (0)
#define HN_FF_WAIT(slot, bar, par) do { HN_FF_T0(); mbar_wait(bar, par); HN_FF_ACC(slot); } while (0)
#define HN_FF_SECTION_BEGIN() const long long ts__ = clock64()
#define HN_FF_SECTION_END(slot) do { if (blockIdx.x == 0 && lane == 0) atomicAdd(&hn_ff_trace[slot], static_cast<unsigned long long>(clock64() - ts__)); } while (0)
#else
#define HN_FF_WAIT(slot, bar, par) mbar_wait(bar, par)
#define HN_FF_SECTION_BEGIN() do { } while (0)
#define HN_FF_SECTION_END(slot) do { } while (0)
#endif

// PW2 = true is the NAS front (stem + the first block's 1x1 expansion, hardnetNAS fbnet_builder.py IRFBlock `pw`): the
// second stage is a pointwise 32 -> 32 conv, i.e. only the centre tap of the same weight image, two N = 32 MMAs per
// tile, no shift-and-add, and the output is plain NHWC ([n][32][32][32]) for the NAS op kernels.
// Second-stage bias as a kernel parameter: parameters live in the constant bank, so `x + bias.v[c]` with a compile-time
// c is one FADD with a constant operand. The former per-tile LDS.128 of the bias were 512 of the ~1400 shared-memory
// data wavefronts per patch of a kernel bound by that pipe.
struct FfBias {
  float v[32];
};

// The kernel body as a device function, shared by front_fused_kernel and front_fused_clip_kernel: CTA `blk` of `nblk` works on
// patches blk, blk + nblk, ...
// CLIP (HardNet variant, TIn = float): there is no patch tensor - `in` is unused and patch clip->n0 + i is cropped around its
// keypoint from the image stack (the reference's clip_patch, FDLNet-master/utils/image_utils.py:11-158, arithmetic in clip.cuh) by
// the stage-1 epilogue warps, which otherwise wait for the stage-1 MMAs most of the time: they fill the raw ring two patches
// ahead, in place of the bulk copies, and the loader warps run unchanged.
template <typename TIn, bool PW2, int FDW, bool CLIP = false>
__device__ __forceinline__ void front_fused_body(const TIn* __restrict__ in, uint16_t* __restrict__ out, const float* __restrict__ w1,
                                                 const float* __restrict__ bias1, const uint4* __restrict__ w2img, const FfBias& bias2,
                                                 int do_norm, int num_patches, int act_bf16, float norm_eps, const CUtensorMap& tm_out,
                                                 const float* __restrict__ dw_w, const float* __restrict__ dw_b, int dw_relu, int fdw_planar,
                                                 const ClipSrc* __restrict__ clip = nullptr) {
  static_assert(FDW == 0 || PW2, "the fused depthwise stage sits behind the pointwise variant");
  static_assert(!CLIP || (sizeof(TIn) == 4 && !PW2), "the cropped patch is fp32 in the raw ring; HardNet variant only");
  constexpr int NACT1 = FDW ? 1 : 2;   // stage-1 activation buffers
  const int blk = static_cast<int>(blockIdx.x), nblk = static_cast<int>(gridDim.x);
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (base - raw_addr);
  const uint32_t a1_addr = base;
  const uint32_t act1_addr = a1_addr + kFfA1;
  const uint32_t w2_addr = act1_addr + NACT1 * kFfAct1;
  const uint32_t w1_addr = w2_addr + kFfW2;
  const uint32_t raw_addr0 = w1_addr + kFfW1;
  const uint32_t stage_addr = raw_addr0 + kFfRaw;                 // FDW: the pointwise output tile (kFfAct2) + depthwise weights
  const uint32_t dww_addr = stage_addr + kFfAct2;
  const uint32_t bar_base = FDW ? dww_addr + kFfDwW + 128 : stage_addr + kFfStage;
  const uint32_t a1_full = bar_base, a1_empty = bar_base + 8, l1_full = bar_base + 16, l1_empty = bar_base + 24;
  auto act1_full = [&](int b) { return bar_base + 32u + 8u * b; };
  auto act1_empty = [&](int b) { return bar_base + 48u + 8u * b; };
  auto c2_full = [&](int a) { return bar_base + 64u + 8u * a; };
  auto c2_empty = [&](int a) { return bar_base + 96u + 8u * a; };
  auto raw_full = [&](int d) { return bar_base + 136u + 8u * d; };
  auto raw_empty = [&](int d) { return bar_base + 168u + 8u * d; };
  auto mma_done = [&](int a) { return bar_base + 200u + 8u * a; };
  const uint32_t tmem_slot = bar_base + 128;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gbase + (tmem_slot - base));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
#ifdef HN_FF_TRACE
  const long long hn_ff_start = clock64();
#endif

  // ---------------------------------------------- one-time setup ----------------------------------------------
  if (warp == kFfIssuer) {
    if (lane == 0) {
      mbar_init(a1_full, 4);    // one arrive per loader warp
      mbar_init(a1_empty, 1);   // tcgen05.commit
      mbar_init(l1_full, 1);    // tcgen05.commit
      mbar_init(l1_empty, 4);   // one arrive per stage-1 epilogue warp
      for (int b = 0; b < 2; ++b) {
        mbar_init(act1_full(b), 4);
        mbar_init(act1_empty(b), PW2 ? 1 : 2);   // tcgen05.commit of every issuing warp
      }
      for (int a = 0; a < 4; ++a) {
        mbar_init(c2_full(a), 1);
        mbar_init(c2_empty(a), 4);
        mbar_init(mma_done(a), 1);
      }
      for (int d = 0; d < kFfRawDepth; ++d) {
        mbar_init(raw_full(d), CLIP ? 4 : 1);   // arrive.expect_tx of the prefetching lane + the copy's complete_tx; CLIP: the four cropping warps
        mbar_init(raw_empty(d), 4);   // one arrive per loader warp
      }
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  } else {
    const int t = threadIdx.x - (warp > kFfIssuer ? 32 : 0);  // dense index over the non-issuer threads
    // conv2 weights: copy the prepared shared-memory image
    for (int i = t; i < static_cast<int>(kFfW2 / 16); i += kFfThreads - 32)
      *reinterpret_cast<uint4*>(gbase + (w2_addr - base) + i * 16) = __ldg(w2img + i);
    // halo rows of both act1 buffers (slots [0, 32) and [33 * 32, 34 * 32) of every plane) are zero and stay zero
    for (int i = t; i < NACT1 * 4 * 2 * 32; i += kFfThreads - 32) {
      const int slot = i & 31, top = (i >> 5) & 1, plane = (i >> 6) & 3, b = i >> 8;
      *reinterpret_cast<uint4*>(gbase + (act1_addr - base) + b * kFfAct1 + plane * kFfPlane +
                                (top ? 33 * 32 + slot : slot) * 16) = make_uint4(0u, 0u, 0u, 0u);
    }
    // stage-1 weights -> canonical no-swizzle [32 x 16] tile: (n/8)*256 + (k/8)*128 + (n%8)*16 + (k%8)*2
    uint16_t* W = reinterpret_cast<uint16_t*>(gbase + (w1_addr - base));
    for (int i = t; i < 32 * 16; i += kFfThreads - 32) {
      const int n = i >> 4, k = i & 15;
      float v = k < 9 ? w1[k * 32 + n] : 0.f;
      if (k == 9 || k == 10) {   // BatchNorm shift as hi + lo against the constant-1 im2col columns
        const float bsh = bias1[n];
        const uint16_t hi = to16bits(bsh, act_bf16);
        const float hif = act_bf16 ? __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(&hi))
                                   : __half2float(*reinterpret_cast<const __half*>(&hi));
        v = k == 9 ? hif : bsh - hif;
      }
      W[((n >> 3) * 256 + (k >> 3) * 128 + (n & 7) * 16 + (k & 7) * 2) >> 1] = to16bits(v, act_bf16);
    }
    if constexpr (FDW == 3 || FDW == 5) {
      __half* dw16 = reinterpret_cast<__half*>(gbase + (dww_addr - base));
      for (int i = t; i < FDW * FDW * 32; i += kFfThreads - 32) dw16[i] = __float2half_rn(dw_w[i]);
      for (int i = t; i < 32; i += kFfThreads - 32) dw16[FDW * FDW * 32 + i] = __float2half_rn(dw_b[i]);
    }
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  // Tensor memory: stage 1 runs in two halves of four 128 x 32 tiles (columns [0, 128)), which leaves room for FOUR
  // 128 x 96 conv2 accumulators (columns [128, 512)): each epilogue group owns two, so the MMAs of its next tile are
  // already done when it finishes the current one.
  const uint32_t tm_l1 = tmem_base;
  const uint32_t tm_c2 = tmem_base + (PW2 ? 256 : 128);   // PW2: stage 1 holds a whole patch (8 x 32 columns)
  constexpr uint32_t C2_STRIDE = PW2 ? 32 : 96;           // accumulator pitch of the second stage

  if (warp >= kFfLoader0 && warp < kFfIssuerB) {
    // ============================== loaders: normalise + im2col of the input patch ==============================
    // Thread = image column x (lane) x 8 consecutive rows (warp): every global load is one coalesced 128 B row segment
    // and every im2col store phase touches 8 consecutive pixels = 8 distinct 16 B bank groups (conflict free).
    // The raw patch comes from a shared-memory ring that one lane keeps kFfRawDepth - 1 patches ahead with bulk async
    // copies, so the HBM latency of the input is off the loaders' critical path.
    const int lw = warp - kFfLoader0;      // rows 8 * lw .. 8 * lw + 7
    const uint32_t one16 = act_bf16 ? 0x3F80u : 0x3C00u;
    constexpr uint32_t RAW_BYTES = 1024 * sizeof(TIn);
    const int n_loc = (num_patches - blk + nblk - 1) / nblk;
    auto prefetch = [&](int j) {           // lane 0 of loader warp 0 only
      const int d = j % kFfRawDepth;
      mbar_wait(raw_empty(d), ((j / kFfRawDepth) & 1) ^ 1u);
      mbar_arrive_expect_tx(raw_full(d), RAW_BYTES);
      const TIn* g = in + (static_cast<size_t>(blk) + static_cast<size_t>(j) * nblk) * 1024;
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                       raw_addr0 + d * 4096), "l"(g), "r"(RAW_BYTES), "r"(raw_full(d))
                   : "memory");
    };
    if (!CLIP && lw == 0 && lane == 0)
      for (int j = 0; j < kFfRawDepth - 1 && j < n_loc; ++j) prefetch(j);
    float* s_red = reinterpret_cast<float*>(gbase + (bar_base + 384 - base));   // [sum | sum of squares][patch parity][4 warps]
    int it = 0;
    for (int patch = blk; patch < num_patches; patch += nblk, ++it) {
      if (!CLIP && lw == 0 && lane == 0 && it + kFfRawDepth - 1 < n_loc) prefetch(it + kFfRawDepth - 1);
      __syncwarp();
      const int d = it % kFfRawDepth;
      HN_FF_WAIT(0, raw_full(d), (it / kFfRawDepth) & 1);
      const TIn* src = reinterpret_cast<const TIn*>(gbase + (raw_addr0 - base) + d * 4096) + lane;
      // 30 branch-free shared-memory loads (clamped addresses, masked afterwards)
      float v[10][3];
      const int xl = lane > 0 ? -1 : 0, xr = lane < 31 ? 1 : 0;
#pragma unroll
      for (int r = 0; r < 10; ++r) {
        const int y = 8 * lw + r - 1;              // warp-uniform
        const TIn* row = src + min(max(y, 0), 31) * 32;
        v[r][0] = static_cast<float>(row[xl]);
        v[r][1] = static_cast<float>(row[0]);
        v[r][2] = static_cast<float>(row[xr]);
      }
      // HardNet.input_norm (hardnet/HardNet.py:306-310): per-patch mean and unbiased std + 1e-7, fused into this load.
      // Every partial sum is a balanced pairwise tree (8 values per lane, xor butterfly over the warp, 2 x 2 warps), so a
      // constant patch has mean == value exactly and normalises to exactly 0, like the reference's 0 / 1e-7.
      float mean = 0.f, inv = 1.f;
      if (do_norm) {
        float* red = s_red + (it & 1) * 4;
        float s8 = ((v[1][1] + v[2][1]) + (v[3][1] + v[4][1])) + ((v[5][1] + v[6][1]) + (v[7][1] + v[8][1]));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s8 += __shfl_xor_sync(0xffffffffu, s8, o);
        if (lane == 0) red[lw] = s8;
        asm volatile("bar.sync 1, 128;" ::: "memory");
        mean = ((red[0] + red[1]) + (red[2] + red[3])) * (1.f / 1024.f);
        float dq[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) { const float dd = v[r + 1][1] - mean; dq[r] = dd * dd; }
        float q8 = ((dq[0] + dq[1]) + (dq[2] + dq[3])) + ((dq[4] + dq[5]) + (dq[6] + dq[7]));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) q8 += __shfl_xor_sync(0xffffffffu, q8, o);
        if (lane == 0) red[8 + lw] = q8;
        asm volatile("bar.sync 1, 128;" ::: "memory");
        const float var = ((red[8] + red[9]) + (red[10] + red[11])) * (1.f / 1023.f);   // torch.std is unbiased
        inv = 1.f / (sqrtf(var) + norm_eps);
      }
#pragma unroll
      for (int r = 0; r < 10; ++r) {
        const int y = 8 * lw + r - 1;
        const bool rowok = y >= 0 && y < 32;       // rows / columns outside the patch are the conv's zero padding
        v[r][0] = (rowok && lane > 0) ? (v[r][0] - mean) * inv : 0.f;
        v[r][1] = rowok ? (v[r][1] - mean) * inv : 0.f;
        v[r][2] = (rowok && lane < 31) ? (v[r][2] - mean) * inv : 0.f;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(raw_empty(d));   // the raw slot may be refilled
      // the stage-1 MMAs of the previous patch must have retired before A1 is overwritten
      HN_FF_WAIT(1, a1_empty, (it & 1) ^ 1u);
      // pixel (y, x): tile y / 4, row r = (y % 4) * 32 + x  ->  (r / 8) * 256 + (r % 8) * 16
      uint8_t* A = gbase + (a1_addr - base) + lw * 2 * 4096 + (lane >> 3) * 256 + (lane & 7) * 16;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        uint4 k0, k1;
        k0.x = pack16_plain(v[j][0], v[j][1], act_bf16);
        k0.y = pack16_plain(v[j][2], v[j + 1][0], act_bf16);
        k0.z = pack16_plain(v[j + 1][1], v[j + 1][2], act_bf16);
        k0.w = pack16_plain(v[j + 2][0], v[j + 2][1], act_bf16);
        k1.x = pack16_plain(v[j + 2][2], 0.f, act_bf16) | (one16 << 16);   // k = 8 (tap 2,2), k = 9: constant 1
        k1.y = one16;                                                       // k = 10: constant 1
        k1.z = 0u; k1.w = 0u;
        uint8_t* dst = A + (j >> 2) * 4096 + (j & 3) * 1024;   // row y = 8 lw + j: tile 2 lw + j / 4, 32-row group j % 4
        *reinterpret_cast<uint4*>(dst) = k0;
        *reinterpret_cast<uint4*>(dst + 128) = k1;
      }
      fence_proxy_async_smem();   // generic-proxy writes -> visible to the tensor core (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(a1_full);
    }
  } else if (warp >= kFfShift0) {
    // ============================== shifters (conv2 only) ==============================
    // D'2 (columns 64..95 of an accumulator) is needed one pixel to the left: tcgen05.shift moves every 32-lane quarter
    // (= one image row) down by one lane, 8 columns per instruction (lane 31 keeps its value and is masked in the
    // epilogue). The shift is NOT ordered behind earlier MMAs by itself, so it waits for the tile's mma_done barrier.
    if constexpr (!PW2) {
      const int g = warp - kFfShift0;
      const int n_local = (num_patches - blk + nblk - 1) / nblk;
      for (int it = 0; it < n_local; ++it) {
#pragma unroll
        for (int tt = 0; tt < 4; ++tt) {
          const int t = 2 * tt + g;
          const int a = t & 3;
          HN_FF_WAIT(7, mma_done(a), (t >> 2) & 1);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t ds = tm_c2 + a * 96 + 64;
#pragma unroll
            for (int c8 = 0; c8 < 4; ++c8) asm volatile("tcgen05.shift.cta_group::1.down [%0];" ::"r"(ds + c8 * 8) : "memory");
            umma_commit(c2_full(a));
          }
          __syncwarp();
        }
      }
    }
  } else if (warp == kFfIssuer || warp == kFfIssuerB) {
    // ============================== UMMA issuers ==============================
    // Descriptor hi words are constants; lo words are `buffer base + compile-time offset` (tile loop fully unrolled).
    const uint32_t idesc1 = make_idesc_f16(kTileM, 32, act_bf16);
    const uint32_t idesc2 = make_idesc_f16(kTileM, PW2 ? 32 : 96, act_bf16);
    constexpr uint32_t L1A_HI = noswizzle_desc_hi(256), L1B_HI = noswizzle_desc_hi(256);
    constexpr uint32_t C2A_HI = noswizzle_desc_hi(128), C2B_HI = noswizzle_desc_hi(512);
    const uint32_t a1_lo = noswizzle_desc_lo(a1_addr, 128);
    const uint32_t b1_lo = noswizzle_desc_lo(w1_addr, 128);
    const uint32_t act_lo0 = noswizzle_desc_lo(act1_addr, kFfPlane);
    const uint32_t w2_lo = noswizzle_desc_lo(w2_addr, 128);
    const int n_local = (num_patches - blk + nblk - 1) / nblk;
    auto issue_l1_half = [&](int half) {
      HN_FF_SECTION_BEGIN();
      if (elect_one()) {
#pragma unroll
        for (int t = 0; t < 4; ++t)
          umma_f16_w(tm_l1 + t * 32, a1_lo + (half * 4 + t) * (4096 >> 4), L1A_HI, b1_lo, L1B_HI, idesc1, 0u);
        if (half == 1) umma_commit(a1_empty);
        umma_commit(l1_full);
      }
      __syncwarp();
      HN_FF_SECTION_END(11);
    };
    const int iw = warp == kFfIssuer ? 0 : 1;
    if constexpr (PW2) {
      if (iw == 0) {
      // The pointwise second stage needs only 4 x 32 accumulator columns, so stage 1 of a WHOLE patch (8 tiles, 256
      // columns) is issued at once and its epilogue drains all eight tiles without waiting for the issuer in between;
      // the pointwise tiles of patch it - 1 are issued behind stage 1 of patch it.
      for (int it = 0; it <= n_local; ++it) {
        if (it < n_local) {
          HN_FF_WAIT(2, a1_full, it & 1);
          if (it > 0) HN_FF_WAIT(3, l1_empty, (it - 1) & 1);   // the epilogue has drained patch it - 1 from tensor memory
          tc_fence_after();
          if (elect_one()) {
#pragma unroll
            for (int t = 0; t < 8; ++t) umma_f16_w(tm_l1 + t * 32, a1_lo + t * (4096 >> 4), L1A_HI, b1_lo, L1B_HI, idesc1, 0u);
            umma_commit(a1_empty);
            umma_commit(l1_full);
          }
          __syncwarp();
        }
        if (it > 0) {
          const int b = FDW ? 0 : (it - 1) & 1;
          HN_FF_WAIT(4, act1_full(b), FDW ? ((it - 1) & 1) : (((it - 1) >> 1) & 1));
          tc_fence_after();
          const uint32_t act_lo = act_lo0 + b * (kFfAct1 >> 4);
#pragma unroll
          for (int t = 0; t < 8; ++t) {
            const int a = t & 3;
            HN_FF_WAIT(6, c2_empty(a), ((t >> 2) & 1) ^ 1u);
            tc_fence_after();
            if (elect_one()) {
              // centre tap only: A = the tile's own 128 slots (image row 4t -> slot (4t + 1) * 32), B = rows [32, 64) of ky = 1
#pragma unroll
              for (int k = 0; k < 2; ++k)
                umma_f16_w(tm_c2 + a * 32, act_lo + (((t * 128 + 32) * 16 + k * 2 * kFfPlane) >> 4), C2A_HI,
                           w2_lo + ((kFfW2Tap + 4 * 512 + k * 256) >> 4), C2B_HI, idesc2, k != 0);
              umma_commit(c2_full(a));
              if (t == 7) umma_commit(act1_empty(b));
            }
            __syncwarp();
          }
        }
      }
      }
    } else {
      // Issuer A (iw = 0) also runs stage 1: the first half of the NEXT patch before tile 0, the second half before
      // tile 4, so the stage-1 epilogue overlaps the conv2 tiles of this patch. Issuer B only issues odd conv2 tiles.
      if (iw == 0 && n_local > 0) {
        mbar_wait(a1_full, 0);
        tc_fence_after();
        issue_l1_half(0);
        mbar_wait(l1_empty, 0);
        tc_fence_after();
        issue_l1_half(1);
      }
      for (int it = 0; it < n_local; ++it) {
        const int b = it & 1;
        const bool more = it + 1 < n_local;
        if (iw == 0 && more) {
          HN_FF_WAIT(2, a1_full, (it + 1) & 1);
          HN_FF_WAIT(3, l1_empty, 1);          // second half of patch `it` has been drained
          tc_fence_after();
          issue_l1_half(0);
        }
        HN_FF_WAIT(4, act1_full(b), (it >> 1) & 1);
        tc_fence_after();
        const uint32_t act_lo = act_lo0 + b * (kFfAct1 >> 4);
#pragma unroll
        for (int tt = 0; tt < 4; ++tt) {
          const int t = 2 * tt + iw;
          if (iw == 0 && tt == 2 && more) {
            HN_FF_WAIT(5, l1_empty, 0);        // first half of patch `it + 1` has been drained
            tc_fence_after();
            issue_l1_half(1);
          }
          const int a = t & 3;             // 8 tiles per patch over 4 buffers: each buffer is used twice per patch
          HN_FF_WAIT(6, c2_empty(a), ((t >> 2) & 1) ^ 1u);
          tc_fence_after();
          HN_FF_SECTION_BEGIN();
          if (elect_one()) {
            const uint32_t d = tm_c2 + a * 96;
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
              for (int k = 0; k < 2; ++k) {
                // A: 128 slots starting at image row 4t + ky - 1 (slot (4t + ky) * 32), channels 16k .. 16k + 15
                umma_f16_w(d, act_lo + (((t * 128 + ky * 32) * 16 + k * 2 * kFfPlane) >> 4), C2A_HI,
                           w2_lo + ((ky * kFfW2Tap + k * 256) >> 4), C2B_HI, idesc2, (ky | k) != 0);
              }
            }
            umma_commit(mma_done(a));                  // -> shifter warp -> c2_full(a)
            if (tt == 3) umma_commit(act1_empty(b));   // this issuer's MMAs no longer read act1[b]
          }
          __syncwarp();
          HN_FF_SECTION_END(13);
        }
      }
    }   // !PW2
  } else if (warp < 4) {
    // ============================== stage-1 epilogue: TMEM -> bias, ReLU, pack -> act1 (smem) ==============================
    const int q = warp;
    int it = 0;
    // CLIP: crop rows 8 q + 4 h .. + 3 of local patch jg into ring slot jg % depth, 16 gathers in flight per thread. A warp-wide
    // load covers a compact 4 x 8 pixel block of the patch, not a row (under rotation a 32-pixel row crosses ~32 image rows; ncu:
    // ~14 sectors per request with blocks). The gathers share the l1tex pipe with the MMAs' operand reads: DESIGN.md section 4.
    // The keypoint of the next patch is fetched as soon as a patch is finished, so its loads are off the next crop's critical path.
    [[maybe_unused]] int jg = 0;
    [[maybe_unused]] ClipKp kp = {};
    [[maybe_unused]] const int n_crop = (num_patches - blk + nblk - 1) / nblk;
    [[maybe_unused]] auto crop_half = [&](int h) {
      if (jg >= n_crop) return;
      const int d = jg % kFfRawDepth;
      if (h == 0) mbar_wait(raw_empty(d), ((jg / kFfRawDepth) & 1) ^ 1u);
      const int prow = 8 * q + 4 * h + (lane >> 3), pcol = lane & 7;   // pixel (prow, 8 r + pcol), r = 0..3
      float* slot = reinterpret_cast<float*>(gbase + (raw_addr0 - base) + d * 4096) + prow * 32 + pcol;
      const bool ok = kp.b >= 0 && kp.b < clip->B;   // image index out of range: NaN patch, like the stand-alone kernel
      const size_t img_off = static_cast<size_t>(ok ? kp.b : 0) * (static_cast<size_t>(clip->H) * clip->W);
      ClipTaps t[4];
      float I[4][4];
#pragma unroll
      for (int r = 0; r < 4; ++r) t[r] = clip_taps(kp, 8 * r + pcol, prow, 32, clip->H, clip->W);
      if (clip->img_u8) {
        const uint8_t* img = static_cast<const uint8_t*>(clip->images) + img_off;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          I[r][0] = clip_pixel(img, t[r].ia); I[r][1] = clip_pixel(img, t[r].ib);
          I[r][2] = clip_pixel(img, t[r].ic); I[r][3] = clip_pixel(img, t[r].id);
        }
      } else {
        const float* img = static_cast<const float*>(clip->images) + img_off;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          I[r][0] = clip_pixel(img, t[r].ia); I[r][1] = clip_pixel(img, t[r].ib);
          I[r][2] = clip_pixel(img, t[r].ic); I[r][3] = clip_pixel(img, t[r].id);
        }
      }
#pragma unroll
      for (int r = 0; r < 4; ++r)
        slot[r * 8] = ok ? clip_blend(t[r], I[r][0], I[r][1], I[r][2], I[r][3]) : __int_as_float(0x7fc00000);
      if (h == 1) {
        __syncwarp();
        if (lane == 0) mbar_arrive(raw_full(d));
        if (++jg < n_crop)
          kp = clip_keypoint(clip->kpts_byxc, clip->kpts_scale, clip->kpts_ori, clip->im_info, clip->kp_per_image,
                             clip->n0 + blk + static_cast<long long>(jg) * nblk);
      }
    };
    if constexpr (CLIP) {
      if (n_crop > 0)
        kp = clip_keypoint(clip->kpts_byxc, clip->kpts_scale, clip->kpts_ori, clip->im_info, clip->kp_per_image, clip->n0 + blk);
      for (int j = 0; j < 2; ++j) { crop_half(0); crop_half(1); }   // two patches ahead of the loaders
    }
    for (int patch = blk; patch < num_patches; patch += nblk, ++it) {
      const int b = FDW ? 0 : it & 1;
      if constexpr (CLIP) crop_half(0);
      HN_FF_WAIT(8, act1_empty(b), (FDW ? (it & 1) : ((it >> 1) & 1)) ^ 1u);
      uint8_t* act = gbase + (act1_addr - base) + b * kFfAct1;
      if constexpr (PW2) {
        HN_FF_WAIT(9, l1_full, it & 1);
        tc_fence_after();
#pragma unroll 2
        for (int t = 0; t < 8; ++t) {
          uint32_t r[32];
          tmem_ld32(tm_l1 + (static_cast<uint32_t>(q * 32) << 16) + t * 32, r);
          tmem_ld_wait();
          uint32_t o[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) o[j] = pack16_relu(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1]), act_bf16);
          uint8_t* dst = act + (t * 128 + q * 32 + lane + 32) * 16;
#pragma unroll
          for (int pl = 0; pl < 4; ++pl)
            *reinterpret_cast<uint4*>(dst + pl * kFfPlane) = make_uint4(o[4 * pl], o[4 * pl + 1], o[4 * pl + 2], o[4 * pl + 3]);
        }
        fence_proxy_async_smem();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(act1_full(b));
          mbar_arrive(l1_empty);
        }
        continue;
      }
#pragma unroll 1
      for (int half = 0; half < 2; ++half) {
        if constexpr (CLIP) { if (half == 1) crop_half(1); }
        HN_FF_WAIT(9, l1_full, half);
        tc_fence_after();
#pragma unroll 1
        for (int tq = 0; tq < 4; ++tq) {
          const int t = half * 4 + tq;
          uint32_t r[32];
          tmem_ld32(tm_l1 + (static_cast<uint32_t>(q * 32) << 16) + tq * 32, r);
          tmem_ld_wait();
          uint32_t o[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) o[j] = pack16_relu(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1]), act_bf16);
          // pixel p = t * 128 + q * 32 + lane  ->  slot p + 32 (one halo row on top)
          uint8_t* dst = act + (t * 128 + q * 32 + lane + 32) * 16;
#pragma unroll
          for (int pl = 0; pl < 4; ++pl)
            *reinterpret_cast<uint4*>(dst + pl * kFfPlane) = make_uint4(o[4 * pl], o[4 * pl + 1], o[4 * pl + 2], o[4 * pl + 3]);
        }
        if (half == 1) fence_proxy_async_smem();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (half == 1) mbar_arrive(act1_full(b));
          mbar_arrive(l1_empty);
        }
      }
    }
  } else {
    // ============================== conv2 epilogue: kx shift-and-add, bias, ReLU, pack -> global ==============================
    const int q = warp & 3;
    const int g = (warp - 4) >> 2;  // this group of four warps owns accumulator buffers g and g + 2
    const uint32_t t_row0 = tm_c2 + (static_cast<uint32_t>(q * 32) << 16);
    const float m_left = lane == 0 ? 0.f : 1.f;     // x - 1 / x + 1 outside the row = the conv's zero padding
    const float m_right = lane == 31 ? 0.f : 1.f;
    for (int patch = blk; patch < num_patches; patch += nblk) {
      uint16_t* opatch = out + static_cast<size_t>(patch) * 32768;
#pragma unroll 1
      for (int tt = 0; tt < 4; ++tt) {
        const int t = 2 * tt + g;
        const int a = t & 3;
        const uint32_t t_row = t_row0 + a * C2_STRIDE;
        HN_FF_WAIT(10, c2_full(a), (t >> 2) & 1);
        tc_fence_after();
        if constexpr (FDW != 0) {
          // pointwise tile -> bias, ReLU, fp16 -> the patch-resident parity-planar tile (pixel (y, x) of plane c at slot
          // ((y & 1) * 2 + (x & 1)) * 256 + (y >> 1) * 16 + (x >> 1)): even / odd lanes write two contiguous 256-byte runs
          uint32_t r[32];
          tmem_ld32(t_row, r);
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(c2_empty(a));
          const uint32_t slot = static_cast<uint32_t>(planar_pixel_slot<32, true>(4 * t + q, lane));
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const uint32_t* rr = r + c * 8;
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stage_addr + c * 16384u + slot * 16u),
                         "r"(pack16_relu(__uint_as_float(rr[0]) + bias2.v[c * 8], __uint_as_float(rr[1]) + bias2.v[c * 8 + 1], 0)),
                         "r"(pack16_relu(__uint_as_float(rr[2]) + bias2.v[c * 8 + 2], __uint_as_float(rr[3]) + bias2.v[c * 8 + 3], 0)),
                         "r"(pack16_relu(__uint_as_float(rr[4]) + bias2.v[c * 8 + 4], __uint_as_float(rr[5]) + bias2.v[c * 8 + 5], 0)),
                         "r"(pack16_relu(__uint_as_float(rr[6]) + bias2.v[c * 8 + 6], __uint_as_float(rr[7]) + bias2.v[c * 8 + 7], 0))
                         : "memory");
          }
          continue;
        }
        if constexpr (PW2) {
          uint32_t r[32];
          tmem_ld32(t_row, r);
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            mbar_arrive(c2_empty(a));
            bulk_wait_read<0>();                  // this warp's previous store is done reading the staging tile
          }
          __syncwarp();
          // A warp's 32 pixels x 32 channels = 2 KB of contiguous NHWC output: staged in the 64B-swizzle pattern (16-byte
          // chunk c of row r at chunk c ^ ((r >> 1) & 3): conflict-free) and written by ONE TMA store. Direct 16-byte
          // stores at a 64-byte stride are 32 sectors per request and kept the L1 pipe of this kernel 79 % busy.
          const uint32_t stg = stage_addr + (warp - 4) * 2048 + lane * 64;
          const uint32_t swz = (lane >> 1) & 3;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const float4 b0 = make_float4(bias2.v[c * 8], bias2.v[c * 8 + 1], bias2.v[c * 8 + 2], bias2.v[c * 8 + 3]);
            const float4 b1 = make_float4(bias2.v[c * 8 + 4], bias2.v[c * 8 + 5], bias2.v[c * 8 + 6], bias2.v[c * 8 + 7]);
            const uint32_t* rr = r + c * 8;
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg + ((c ^ swz) << 4)),
                         "r"(pack16_relu(__uint_as_float(rr[0]) + b0.x, __uint_as_float(rr[1]) + b0.y, act_bf16)),
                         "r"(pack16_relu(__uint_as_float(rr[2]) + b0.z, __uint_as_float(rr[3]) + b0.w, act_bf16)),
                         "r"(pack16_relu(__uint_as_float(rr[4]) + b1.x, __uint_as_float(rr[5]) + b1.y, act_bf16)),
                         "r"(pack16_relu(__uint_as_float(rr[6]) + b1.z, __uint_as_float(rr[7]) + b1.w, act_bf16))
                         : "memory");
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&tm_out, stage_addr + (warp - 4) * 2048, 0, patch * 1024 + (4 * t + q) * 32);
            bulk_commit();
          }
          continue;
        }
        // channel-planar parity layout for the stride-2 conv3: [plane][ypar][xpar][16][16][8]
        uint4* dst = reinterpret_cast<uint4*>(opatch) + planar_pixel_slot<32, true>(4 * t + q, lane);
        // six TMEM loads (two 8-channel chunks) are in flight per wait: half the exposed round trips of a per-chunk wait
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2) {
        uint32_t r0[2][8], r1[2][8], r2[2][8];
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          tmem_ld8(t_row + (2 * h2 + cc) * 8, r0[cc]);
          tmem_ld8(t_row + 32 + (2 * h2 + cc) * 8, r1[cc]);
          tmem_ld8(t_row + 64 + (2 * h2 + cc) * 8, r2[cc]);
        }
        tmem_ld_wait();
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          const int c = 2 * h2 + cc;
          const float bias[8] = {bias2.v[c * 8], bias2.v[c * 8 + 1], bias2.v[c * 8 + 2], bias2.v[c * 8 + 3],
                                 bias2.v[c * 8 + 4], bias2.v[c * 8 + 5], bias2.v[c * 8 + 6], bias2.v[c * 8 + 7]};
          // The left neighbour's partial sum crosses lanes as fp16 pairs: one shuffle moves two values (shuffles run on
          // the shared-memory pipe, the busiest unit of this kernel). |D'| stays far inside the fp16 range and the extra
          // rounding (2^-11 relative on one addend) is below the output's own 16-bit rounding. Sums are fp32.
          float v[8];
#pragma unroll
          for (int j = 0; j < 8; j += 2) {
            const uint32_t lp = __shfl_up_sync(0xffffffffu, pack16_plain(__uint_as_float(r0[cc][j]), __uint_as_float(r0[cc][j + 1]), 0), 1);
            const float2 lf = __half22float2(*reinterpret_cast<const __half2*>(&lp));    // D'0 of pixel x - 1
            // r2 already holds D'2 of pixel x + 1 (shifted in tensor memory by the issuer)
            v[j] = fmaf(__uint_as_float(r2[cc][j]), m_right, fmaf(lf.x, m_left, __uint_as_float(r1[cc][j]) + bias[j]));
            v[j + 1] = fmaf(__uint_as_float(r2[cc][j + 1]), m_right, fmaf(lf.y, m_left, __uint_as_float(r1[cc][j + 1]) + bias[j + 1]));
          }
          dst[c * 1024] = make_uint4(pack16_relu(v[0], v[1], act_bf16), pack16_relu(v[2], v[3], act_bf16),
                                     pack16_relu(v[4], v[5], act_bf16), pack16_relu(v[6], v[7], act_bf16));
        }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(c2_empty(a));
      }
      if constexpr (FDW != 0) {
        // ---- stride-2 depthwise conv / max-pool of the patch-resident tile by the same eight warps: a thread owns 8
        // channels x one output column x a strip of 4 output rows (4 planes x 16 columns x 4 strips = 256 items) ----
        {
          HN_FF_SECTION_BEGIN();
          asm volatile("bar.sync 2, 256;" ::: "memory");          // all eight tiles of this patch are in the tile
          HN_FF_SECTION_END(17);
        }
        {
          HN_FF_SECTION_BEGIN();
          constexpr int K = FDW == 1 ? 3 : FDW, PAD = K >> 1, SH = 4, NR = (SH - 1) * 2 + K;
          const int item = static_cast<int>(threadIdx.x) - 128;   // warps 4..11
          const int ox = item & 15, ys = (item >> 4) & 3, plane = item >> 6;
          const uint8_t* tile = gbase + (stage_addr - base) + plane * 16384;
          const __half* s_dw = reinterpret_cast<const __half*>(gbase + (dww_addr - base));
          const uint32_t ninf = 0xFC00FC00u;
          __half2 acc[SH][4];
          if constexpr (FDW == 1) {
#pragma unroll
            for (int j = 0; j < SH; ++j)
#pragma unroll
              for (int qq = 0; qq < 4; ++qq) acc[j][qq] = *reinterpret_cast<const __half2*>(&ninf);
          } else {
            const uint4 b = *reinterpret_cast<const uint4*>(s_dw + K * K * 32 + plane * 8);
#pragma unroll
            for (int j = 0; j < SH; ++j) {
              acc[j][0] = *reinterpret_cast<const __half2*>(&b.x); acc[j][1] = *reinterpret_cast<const __half2*>(&b.y);
              acc[j][2] = *reinterpret_cast<const __half2*>(&b.z); acc[j][3] = *reinterpret_cast<const __half2*>(&b.w);
            }
          }
          const int iy0 = ys * SH * 2 - PAD;
#pragma unroll
          for (int kx = 0; kx < K; ++kx) {
            const int ix = ox * 2 + kx - PAD;
            const bool x_ok = ix >= 0 && ix < 32;
            uint4 wk[K];
            if constexpr (FDW != 1) {
#pragma unroll
              for (int ky = 0; ky < K; ++ky) wk[ky] = *reinterpret_cast<const uint4*>(s_dw + (ky * K + kx) * 32 + plane * 8);
            }
#pragma unroll
            for (int r = 0; r < NR; ++r) {
              const int iy = iy0 + r;
              const bool ok = x_ok && iy >= 0 && iy < 32;
              uint4 xv = FDW == 1 ? make_uint4(ninf, ninf, ninf, ninf) : make_uint4(0u, 0u, 0u, 0u);
              if (ok) xv = *reinterpret_cast<const uint4*>(tile + planar_pixel_slot<32, true>(iy, ix) * 16);
              const __half2 x[4] = {*reinterpret_cast<const __half2*>(&xv.x), *reinterpret_cast<const __half2*>(&xv.y),
                                    *reinterpret_cast<const __half2*>(&xv.z), *reinterpret_cast<const __half2*>(&xv.w)};
#pragma unroll
              for (int j = 0; j < SH; ++j) {
                const int ky = r - j * 2;          // compile-time after unrolling
                if (ky >= 0 && ky < K) {
                  if constexpr (FDW == 1) {
#pragma unroll
                    for (int qq = 0; qq < 4; ++qq) acc[j][qq] = __hmax2_nan(acc[j][qq], x[qq]);
                  } else {
                    const __half2 wv[4] = {*reinterpret_cast<const __half2*>(&wk[ky].x), *reinterpret_cast<const __half2*>(&wk[ky].y),
                                           *reinterpret_cast<const __half2*>(&wk[ky].z), *reinterpret_cast<const __half2*>(&wk[ky].w)};
#pragma unroll
                    for (int qq = 0; qq < 4; ++qq) acc[j][qq] = __hfma2(x[qq], wv[qq], acc[j][qq]);
                  }
                }
              }
            }
          }
          uint16_t* optr = fdw_planar ? out + static_cast<size_t>(patch) * 8192 + plane * 2048 + ((ys * SH) * 16 + ox) * 8
                                      : out + (static_cast<size_t>(patch) * 256 + (ys * SH) * 16 + ox) * 32 + plane * 8;
          const int orow = fdw_planar ? 16 * 8 : 16 * 32;
          const __half2 hzero = __float2half2_rn(0.f);
#pragma unroll
          for (int j = 0; j < SH; ++j) {
            if (FDW != 1 && dw_relu) {
#pragma unroll
              for (int qq = 0; qq < 4; ++qq) acc[j][qq] = __hmax2(acc[j][qq], hzero);
            }
            *reinterpret_cast<uint4*>(optr + j * orow) =
                make_uint4(*reinterpret_cast<const uint32_t*>(&acc[j][0]), *reinterpret_cast<const uint32_t*>(&acc[j][1]),
                           *reinterpret_cast<const uint32_t*>(&acc[j][2]), *reinterpret_cast<const uint32_t*>(&acc[j][3]));
          }
          HN_FF_SECTION_END(14);
        }
        {
          HN_FF_SECTION_BEGIN();
          asm volatile("bar.sync 2, 256;" ::: "memory");          // the tile may be overwritten by the next patch
          HN_FF_SECTION_END(18);
        }
      }
    }
  }

  if constexpr (PW2 && FDW == 0) {
    if (warp >= 4 && warp < kFfIssuer && lane == 0) bulk_wait_all<0>();   // output stores still read this CTA's smem
  }
  tc_fence_before();
  __syncthreads();
#ifdef HN_FF_TRACE
  if (blk == 0 && threadIdx.x == 0) {
    atomicAdd(&hn_ff_trace[15], static_cast<unsigned long long>(clock64() - hn_ff_start));
    atomicAdd(&hn_ff_trace[16], static_cast<unsigned long long>((num_patches + nblk - 1) / nblk));
  }
#endif
  if (warp == kFfIssuer) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// FDW: 0 = none; 3 / 5 = depthwise 3x3 / 5x5 stride 2 (+ bias, optional ReLU) behind the pointwise stage; 1 = MaxPool 3x3
// stride 2 pad 1 (hardnetNAS fbnet_builder.py:455-570 IRFBlock `dw`, :202-228 Identity). fp16 activations only.
template <typename TIn, bool PW2 = false, int FDW = 0>
__global__ void __launch_bounds__(kFfThreads, 1)
front_fused_kernel(const TIn* __restrict__ in, uint16_t* __restrict__ out /*[n][4 planes][2][2][16][16][8]; PW2: NHWC; FDW: NHWC [n][16][16][32]*/,
                   const float* __restrict__ w1 /*[9][32] folded*/, const float* __restrict__ bias1 /*[32]*/,
                   const uint4* __restrict__ w2img /*kFfW2 bytes, shared-memory image*/,
                   const __grid_constant__ FfBias bias2 /*[32]*/, int do_norm /*0: no input normalisation*/,
                   int num_patches, int act_bf16, float norm_eps /*added to the std: 1e-7 HardNet, 1e-8 HardNetNeiMask*/,
                   const __grid_constant__ CUtensorMap tm_out /*PW2: [n * 1024, 32] as 32 x 32 boxes, 64B swizzle*/,
                   const float* __restrict__ dw_w = nullptr /*FDW 3 | 5: [k * k][32] folded*/, const float* __restrict__ dw_b = nullptr /*[32]*/,
                   int dw_relu = 0, int fdw_planar = 0 /*FDW output channel-planar [n][4][16][16][8] (the tail kernel's bulk-copy layout)*/) {
  front_fused_body<TIn, PW2, FDW>(in, out, w1, bias1, w2img, bias2, do_norm, num_patches, act_bf16, norm_eps, tm_out, dw_w, dw_b, dw_relu,
                                  fdw_planar);
}

// The HardNet front kernel fed by clip_patch on the fly (hn_forward_clip): same stages, patches cropped inside the kernel.
__global__ void __launch_bounds__(kFfThreads, 1)
front_fused_clip_kernel(const __grid_constant__ ClipSrc clip, uint16_t* __restrict__ out, const float* __restrict__ w1,
                        const float* __restrict__ bias1, const uint4* __restrict__ w2img, const __grid_constant__ FfBias bias2,
                        int num_patches, int act_bf16, float norm_eps, const __grid_constant__ CUtensorMap tm_out) {
  front_fused_body<float, false, 0, true>(nullptr, out, w1, bias1, w2img, bias2, 1, num_patches, act_bf16, norm_eps, tm_out, nullptr,
                                          nullptr, 0, 0, &clip);
}

}  // namespace hn
