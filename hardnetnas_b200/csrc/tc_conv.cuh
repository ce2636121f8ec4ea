// Shared pieces of the tcgen05 kernels (parameter block, 16-bit packing, channel-planar addressing) and the descriptor head:
//
//   gemm_l2norm_kernel : the 8x8 head conv (features[19..20] + L2Norm, HardNet.py:300-301,314-315 and
//     Utils.py:19-22) as a [B, K] x [K, 128] GEMM with bias + L2-normalise in the epilogue (also the NAS
//     head with K = 2048).
//
// Roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM owner + UMMA issuer, warps 2..5 = epilogue
// (TMEM -> registers -> bias / L2-normalise -> global). The producer / issuer loops run warp-uniformly (every lane
// executes the control flow, elect.sync picks the lane that issues), which lets the compiler keep the loop state in
// uniform registers. Two accumulator buffers in TMEM let the epilogue of tile i overlap the MMAs of tile i+1.
// The 3x3 convs run on the CTA-pair kernel of tc_conv_pair.cuh.
#pragma once

#include "common.cuh"

namespace hn {

constexpr int kTileM = 128;
constexpr int kTcThreads = 192;

enum : int { DT_F32 = 0, DT_F16 = 1, DT_BF16 = 2, DT_U8 = 3, DT_F8E4M3 = 5 };   // = hn_dtype

struct TcParams {
  CUtensorMap tmA[4];      // conv stride 1 / gemm: [0]; conv stride 2: parity views [ypar * 2 + xpar]
  CUtensorMap tmB;         // weights, [C_out, K] K-major
  const float* bias;       // [N] folded BatchNorm shift
  float bias_v[128];       // conv kernels: the same values BY VALUE - parameters sit in the constant bank, so the epilogue's
                           // `acc + bias` is an FADD with a constant operand instead of shared-memory loads on the busy L1 pipe
  void* out;               // conv: 16-bit channel-planar (see above); head: f32/f16/bf16/e4m3 [rows, N]
  long long total_rows;    // valid output rows (pixels or patches)
  int num_tiles;
  int num_k_stages;        // gemm only: K / (G * 64)
  int act_bf16;            // 16-bit activation flavour: 0 = fp16, 1 = bf16
  int out_dtype;           // head only: DT_F32 / DT_F16 / DT_BF16 / DT_F8E4M3
  float l2_eps;            // head only: 1e-10 (Utils.py:18); 0 for the NAS head
  int k_splits;            // head only: > 1 = split-K (small batches): a CTA reduces num_k_stages / k_splits stages of one row tile
                           // and writes raw fp32 partial sums to `partial`; head_finalize_kernel adds them, the bias and the norm
  float* partial;          // [k_splits][num_tiles * 128][128] fp32
};

// Parameters of the fused conv3 + conv4 kernel (tc_conv34.cuh)
struct Conv34Params {
  CUtensorMap tmA[4];   // conv2 output, parity views [ypar * 2 + xpar], box (16 px * 8, 9 rows, 1 patch, 4 planes)
  CUtensorMap tmB3;     // conv3 weights [64][9 * 32], box (32, 32 rows), 64B swizzle
  CUtensorMap tmB4;     // conv4 weights [64][9 * 64], box (64, 32 rows), 128B swizzle
  float bias3[64];      // folded BN shifts, by value (constant bank)
  float bias4[64];
  void* out;            // conv4 output, channel-planar parity layout [patch][8 planes][ypar][xpar][8][8][8]
  int n_patches;
  int act_bf16;
};

__device__ __forceinline__ uint32_t pack16(float lo, float hi, int bf16) {
  if (bf16) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  }
  // saturate instead of producing inf for out-of-range activations
  lo = fminf(lo, 65504.f);
  hi = fminf(hi, 65504.f);
  __half2 v = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

constexpr uint32_t tmem_cols_for(int n) {
  return (2 * n <= 32) ? 32u : (2 * n <= 64) ? 64u : (2 * n <= 128) ? 128u : (2 * n <= 256) ? 256u : 512u;
}

__device__ __forceinline__ uint64_t make_noswizzle_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(lbo_bytes >> 4) << 16;   // K direction: next 8-channel core matrix
  d |= static_cast<uint64_t>(sbo_bytes >> 4) << 32;   // M/N direction: next 8-row core matrix
  d |= 1ull << 46;
  return d;  // layout type 0 = no swizzle
}

// Element offset of pixel (y, x) inside one 8-channel plane of a W x W image (units of 8-channel groups).
template <int W, bool PARITY>
__device__ __forceinline__ int planar_pixel_slot(int y, int x) {
  if (PARITY) return ((y & 1) * 2 + (x & 1)) * (W * W / 4) + (y >> 1) * (W / 2) + (x >> 1);
  return y * W + x;
}

// {lo, hi} -> two 16-bit values with ReLU and saturation to the largest finite value, one instruction (F2FP.SATFINITE.RELU)
__device__ __forceinline__ uint32_t pack16_relu(float lo, float hi, int bf16) {
  uint32_t r;
  if (bf16) asm("cvt.rn.relu.satfinite.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  else asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t pack16_plain(float lo, float hi, int bf16) {
  uint32_t r;
  if (bf16) asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  else asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// ------------------------------------------------------------------------------------------------------------
// [rows, K] x [K, 128] GEMM + bias + L2 normalisation (descriptor head)
// ------------------------------------------------------------------------------------------------------------
constexpr int kHeadN = 128;
constexpr int kHeadG = 2;        // two 64-wide k-blocks per stage
constexpr int kHeadStages = 3;
constexpr uint32_t kHeadBlk = kTileM * 128;  // one 128 x 64 fp16 operand tile
constexpr size_t kHeadSmem = size_t(kHeadStages) * kHeadG * 2 * kHeadBlk + 1024 + 256 + kHeadN * 4;

// TILES = 2 (bulk batches, no split-K): a work item is two consecutive 128-row tiles that share every streamed weight block.
// At the bulk rate all 148 CTAs stream the same 2 MB of weights out of L2 per tile next to 2 MB of activations - the kernel is
// bound by that traffic (32 KB per patch through the L2 -> SM fabric for 1 MMAC per patch); two tiles per weight stream make it 24 KB.
template <int N, int TILES = 1>
__global__ void __launch_bounds__(kTcThreads, 1) gemm_l2norm_kernel(const __grid_constant__ TcParams p) {
  constexpr int STAGES = TILES == 2 ? 2 : kHeadStages, G = kHeadG;
  static_assert(N == kHeadN, "descriptor head is 128 wide");
  static_assert(TILES == 1 || TILES == 2, "one or two row tiles per work item");
  constexpr uint32_t STAGE_BYTES = G * (TILES + 1) * kHeadBlk;   // per k-block: TILES activation tiles + one weight tile
  static_assert(size_t(STAGES) * STAGE_BYTES + 1024 + 256 + kHeadN * 4 <= kHeadSmem, "shared memory budget");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  const uint32_t bar_base = base + STAGES * STAGE_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 4);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw_addr));
  float* s_bias = reinterpret_cast<float*>(smem_raw + (bar_base + 256u - raw_addr));
  constexpr uint32_t TMEM_COLS = tmem_cols_for(TILES * N);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmA[0]);
    tma_prefetch_desc(&p.tmB);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < STAGES; ++s) {
        mbar_init(full_bar(s), 1);
        mbar_init(empty_bar(s), 1);
      }
      for (int a = 0; a < 2; ++a) {
        mbar_init(tfull_bar(a), 1);
        mbar_init(tempty_bar(a), 4);
      }
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, TMEM_COLS);
    tmem_relinquish();
  }
  if (warp >= 2) {
    for (int i = threadIdx.x - 64; i < N; i += 128) s_bias[i] = p.bias[i];
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    int stage = 0;
    uint32_t phase = 0;
    const int splits = (TILES == 1 && p.k_splits > 1) ? p.k_splits : 1;
    const int nks = p.num_k_stages / splits;                 // k-stages per work item
    const int n_items = TILES == 2 ? (p.num_tiles + 1) / 2 : p.num_tiles * splits;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const int tile = TILES == 2 ? item * 2 : item / splits, ks0 = TILES == 2 ? 0 : (item - tile * splits) * nks;
#pragma unroll 1
      for (int ksi = 0; ksi < nks; ++ksi) {
        const int ks = ks0 + ksi;
        mbar_wait(empty_bar(stage), phase ^ 1u);
        if (elect_one()) {
          const uint32_t st_base = base + stage * STAGE_BYTES;
          mbar_arrive_expect_tx(full_bar(stage), STAGE_BYTES);
#pragma unroll
          for (int g = 0; g < G; ++g) {
#pragma unroll
            for (int tl = 0; tl < TILES; ++tl)   // a tile past the end of the batch reads out-of-range rows: TMA zero-fills them
              tma_load_2d(st_base + (g * TILES + tl) * kHeadBlk, &p.tmA[0], full_bar(stage), (ks * G + g) * 64, (tile + tl) * kTileM);
            tma_load_2d(st_base + (G * TILES + g) * kHeadBlk, &p.tmB, full_bar(stage), (ks * G + g) * 64, 0);
          }
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc = make_idesc_f16(kTileM, N, p.act_bf16);
    constexpr uint32_t HI = kmajor_desc_hi(128);
    const uint32_t ring_lo = kmajor_desc_lo(base);
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    const int splits = (TILES == 1 && p.k_splits > 1) ? p.k_splits : 1;
    const int nks = p.num_k_stages / splits;
    const int n_items = TILES == 2 ? (p.num_tiles + 1) / 2 : p.num_tiles * splits;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * (TILES * N);
#pragma unroll 1
      for (int ks = 0; ks < nks; ++ks) {
        mbar_wait(full_bar(stage), phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t lo = ring_lo + static_cast<uint32_t>(stage) * (STAGE_BYTES >> 4);
#pragma unroll
          for (int g = 0; g < G; ++g) {
#pragma unroll
            for (int tl = 0; tl < TILES; ++tl) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_f16_w(d_tmem + tl * N, lo + (((g * TILES + tl) * kHeadBlk) >> 4) + 2u * k, HI,
                           lo + (((G * TILES + g) * kHeadBlk) >> 4) + 2u * k, HI, idesc, (ks | g | k) != 0);
            }
          }
          umma_commit(empty_bar(stage));
          if (ks == nks - 1) umma_commit(tfull_bar(acc));
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else {
    const int q = warp & 3;
    const int row_in_tile = q * 32 + lane;
    int it = 0;
    const int splits = (TILES == 1 && p.k_splits > 1) ? p.k_splits : 1;
    const int n_items = TILES == 2 ? (p.num_tiles + 1) / 2 : p.num_tiles * splits;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
#pragma unroll 1
      for (int tl = 0; tl < TILES; ++tl) {
      const int tile = TILES == 2 ? item * 2 + tl : item / splits, split = TILES == 2 ? 0 : item - tile * splits;
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * (TILES * N) + tl * N;
      const long long row = static_cast<long long>(tile) * kTileM + row_in_tile;
      const bool valid = row < p.total_rows;
      if (splits > 1) {
        // split-K: raw partial sums of this K range; bias, norm and the output type belong to head_finalize_kernel
        float* dstp = p.partial + (static_cast<long long>(split) * p.num_tiles * kTileM + row) * N;
#pragma unroll
        for (int c0 = 0; c0 < N; c0 += 32) {
          uint32_t r[32];
          tmem_ld32(t_row + c0, r);
          tmem_ld_wait();
          if (valid) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              reinterpret_cast<float4*>(dstp + c0)[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]),
                                                                    __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3]));
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(acc));
        continue;   // (TILES == 1 on this path: the tile loop has one trip)
      }
      // bias, then x / sqrt(sum(x*x) + eps) over the N columns of the row (Utils.py:19-22)
      float ss = 0.f;
#pragma unroll
      for (int c0 = 0; c0 < N; c0 += 32) {
        uint32_t r[32];
        tmem_ld32(t_row + c0, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float v = __uint_as_float(r[j]) + s_bias[c0 + j];
          ss = fmaf(v, v, ss);
        }
      }
      const float inv = 1.0f / sqrtf(ss + p.l2_eps);
#pragma unroll
      for (int c0 = 0; c0 < N; c0 += 32) {
        uint32_t r[32];
        tmem_ld32(t_row + c0, r);
        tmem_ld_wait();
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = (__uint_as_float(r[j]) + s_bias[c0 + j]) * inv;
        if (valid) {
          if (p.out_dtype == DT_F32) {
            float4* dst = reinterpret_cast<float4*>(static_cast<float*>(p.out) + row * N + c0);
#pragma unroll
            for (int j = 0; j < 8; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          } else if (p.out_dtype == DT_F8E4M3) {
            uint4* dst = reinterpret_cast<uint4*>(static_cast<uint8_t*>(p.out) + row * N + c0);
#pragma unroll
            for (int j = 0; j < 2; ++j)
              dst[j] = make_uint4(pack_e4m3x4(v[16 * j], v[16 * j + 1], v[16 * j + 2], v[16 * j + 3]),
                                  pack_e4m3x4(v[16 * j + 4], v[16 * j + 5], v[16 * j + 6], v[16 * j + 7]),
                                  pack_e4m3x4(v[16 * j + 8], v[16 * j + 9], v[16 * j + 10], v[16 * j + 11]),
                                  pack_e4m3x4(v[16 * j + 12], v[16 * j + 13], v[16 * j + 14], v[16 * j + 15]));
          } else {
            uint4* dst = reinterpret_cast<uint4*>(static_cast<uint16_t*>(p.out) + row * N + c0);
            const int bf = p.out_dtype == DT_BF16;
#pragma unroll
            for (int j = 0; j < 4; ++j)
              dst[j] = make_uint4(pack16(v[8 * j], v[8 * j + 1], bf), pack16(v[8 * j + 2], v[8 * j + 3], bf),
                                  pack16(v[8 * j + 4], v[8 * j + 5], bf), pack16(v[8 * j + 6], v[8 * j + 7], bf));
          }
        }
      }
      }   // tile loop
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// Second half of the split-K head: sum the K-range partials in split order, add the bias, L2-normalise, store.
// One warp per descriptor row, a lane owns 4 of the 128 columns.
static __global__ void __launch_bounds__(256) head_finalize_kernel(const float* __restrict__ partial, int k_splits, long long rows_padded,
                                                            long long total_rows, const float* __restrict__ bias, float l2_eps,
                                                            void* __restrict__ out, int out_dtype) {
  const long long row = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= total_rows) return;
  float4 v = *reinterpret_cast<const float4*>(bias + lane * 4);
  for (int s = 0; s < k_splits; ++s) {
    const float4 a = *reinterpret_cast<const float4*>(partial + (static_cast<long long>(s) * rows_padded + row) * 128 + lane * 4);
    v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
  }
  float ss = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, v.w * v.w)));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float inv = 1.0f / sqrtf(ss + l2_eps);
  v.x *= inv; v.y *= inv; v.z *= inv; v.w *= inv;
  if (out_dtype == DT_F32) {
    *reinterpret_cast<float4*>(static_cast<float*>(out) + row * 128 + lane * 4) = v;
  } else if (out_dtype == DT_F8E4M3) {
    *reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(out) + row * 128 + lane * 4) = pack_e4m3x4(v.x, v.y, v.z, v.w);
  } else {
    const int bf = out_dtype == DT_BF16;
    *reinterpret_cast<uint2*>(static_cast<uint16_t*>(out) + row * 128 + lane * 4) = make_uint2(pack16(v.x, v.y, bf), pack16(v.z, v.w, bf));
  }
}

}  // namespace hn
