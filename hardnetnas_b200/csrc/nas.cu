// NAS-derived descriptor nets (hardnetNAS/fbnet_building_blocks/fbnet_builder.py + the supernet stem/head of
// hardnetNAS/supernet_functions/model_supernet.py:57-58,64-68,84) behind the C ABI.
//
// The Python side compiles the module tree into a flat op list (BatchNorm folded, channel shuffle folded into
// the producing 1x1 conv, grouped 1x1 convs expanded to block-diagonal dense matrices). Here every op is one
// kernel over a chunk of patches, activations NHWC 16-bit in three handle-owned slots:
//   STEM    conv 3x3 1->32 + BN + ReLU                  l1_norm_conv_kernel (no input normalisation)
//   PW      1x1 conv + BN [+ReLU] [+residual]           pw_gemm_kernel: tcgen05 GEMM [pixels, C_in] x [C_in, C_out]
//   DW      depthwise k3/k5, stride 1/2 + BN + ReLU     dw_conv_kernel (CUDA cores, 8 channels per thread)
//   MAXPOOL 3x3 stride 2 pad 1                          maxpool_kernel
//   SE      x * sigmoid(fc2(relu(fc1(avgpool(x)))))     se_kernel (one CTA per patch)
//   HEAD    k x k full conv -> 128 + BN + y/||y||       gemm_l2norm_kernel (eps = 0, like torch.norm)
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "handle.h"
#include "host_common.h"
#include "tc_conv.cuh"
#include "nas_tail.cuh"

namespace hn {

enum : int { OP_STEM = 0, OP_PW = 1, OP_DW = 2, OP_MAXPOOL = 3, OP_SE = 4, OP_HEAD = 5 };

// ------------------------------------------------------------------------------------------------------------
// pointwise (1x1) convolution as a tensor-core GEMM
// ------------------------------------------------------------------------------------------------------------
struct PwParams {
  CUtensorMap tmA;       // activations [rows, C_in]
  CUtensorMap tmB;       // weights [C_out, C_in] (BN scale folded)
  CUtensorMap tmO;       // output [rows, C_out] as 32-row x min(NT, 64)-column swizzled store boxes
  CUtensorMap tmR;       // residual (same geometry as tmO), loaded into the output staging tile by the epilogue
  const float* bias;     // [C_out]
  const uint16_t* res;   // optional residual [rows, C_out]
  uint16_t* out;         // [rows, C_out]
  long long total_rows;
  int num_tiles;         // m_tiles * n_tiles
  int n_tiles;
  int num_kb;            // C_in / (KCB / 2)
  int cout;              // output row length as the kernel sees it (2 x C_out for row-paired ops)
  int bias_n;            // length of `bias` (the kernel indexes it modulo this)
  int nt, kcb;           // kernel configuration
  int row_div;           // 2 when two consecutive rows are processed as one (C_in = 32), else 1
  int relu;
  int act_bf16;
};

// A 32-channel activation row is 64 bytes; TMA loads and stores of 64-byte rows ran these ops at ~3.8 TB/s where the
// same kernel moves 128-byte rows at > 5 TB/s. Rows of a C_in = 32 op are therefore processed in PAIRS: [rows, 32] is
// viewed as [rows / 2, 64] (the NHWC tensor is contiguous, rows per patch are even) and the weight becomes the block
// diagonal [[W, 0], [0, W]], so the output [rows / 2, 2 C_out] is the same memory as [rows, C_out]. The extra zero MACs
// are free (the tensor pipe idles in these HBM-bound ops).
static bool pw_row_paired(const hn_nas_op& o) { return o.cin == 32 && o.cout <= 128; }

// A pointwise stage is small (8-16 KB of activations + the weight tile), so the ring is DEEP: the bytes in flight per SM,
// not the tensor pipe, set the rate of these HBM-bound GEMMs (4 stages left them at ~3.3 TB/s).
// Warps: 0 TMA producer, 1 TMEM owner + UMMA issuer, then GROUPS epilogue groups of four warps that take tiles round
// robin (one tile's TMEM -> bias/ReLU -> store chain is ~1000 cycles of mostly latency; a single group left these
// HBM-bound kernels at ~3.5 TB/s). Four accumulators, tile `it` uses accumulator it % 4.
template <int NT>
constexpr int pw_groups() { return NT <= 64 ? 4 : 2; }
template <int NT>
constexpr int pw_threads() { return 64 + 128 * pw_groups<NT>(); }
// Output staging for the swizzled TMA stores: one (32 rows x NT columns) buffer per epilogue warp; NT = 96 keeps the
// direct stores (its rows do not split into equal power-of-two boxes).
template <int NT>
constexpr bool pw_tma_out() { return NT == 32 || NT == 64 || NT == 128; }
template <int NT>
constexpr uint32_t pw_staging_bytes() { return pw_tma_out<NT>() ? 4u * pw_groups<NT>() * 32u * NT * 2u : 0u; }
template <int NT, int KCB>
constexpr int pw_stages() {
  constexpr int s = (220 * 1024 - static_cast<int>(pw_staging_bytes<NT>())) / (kTileM * KCB + NT * KCB);
  return s > 16 ? 16 : s;
}
template <int NT, int KCB>
constexpr uint32_t pw_bias_off() { return (8u * (2 * pw_stages<NT, KCB>() + 9 + 16) + 15u) & ~15u; }   // + 16 residual barriers

template <int NT, int KCB>
constexpr size_t pw_smem_bytes() {
  return size_t(pw_stages<NT, KCB>()) * (size_t(kTileM) * KCB + size_t(NT) * KCB) + pw_staging_bytes<NT>() + 1024 +
         pw_bias_off<NT, KCB>() + 512 * 4;
}

__device__ __forceinline__ float2 unpack16(uint32_t v, int bf16) {
  if (bf16) {
    return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v));
  }
  return __half22float2(*reinterpret_cast<const __half2*>(&v));
}

template <int NT, int KCB>
__global__ void __launch_bounds__(pw_threads<NT>(), 1) pw_gemm_kernel(const __grid_constant__ PwParams p) {
  constexpr int GROUPS = pw_groups<NT>();
  constexpr int STAGES = pw_stages<NT, KCB>();
  constexpr uint32_t A_BYTES = kTileM * KCB;
  constexpr uint32_t B_BYTES = NT * KCB;
  constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr uint32_t TMEM_COLS = tmem_cols_for(2 * NT);   // four NT-column accumulators
  constexpr int KC = KCB / 2;
  static_assert(B_BYTES % 1024 == 0, "weight tile must stay 1024B aligned");

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  const uint32_t staging_base = base + STAGES * STAGE_BYTES;            // 1024-byte aligned (stage sizes are multiples)
  const uint32_t bar_base = staging_base + pw_staging_bytes<NT>();
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 4 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 8);
  auto res_bar = [&](int w) { return bar_base + 8u * (2 * STAGES + 9 + w); };   // one per epilogue warp
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw_addr));
  float* s_bias = reinterpret_cast<float*>(smem_raw + (bar_base + pw_bias_off<NT, KCB>() - raw_addr));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmA);
    tma_prefetch_desc(&p.tmB);
    tma_prefetch_desc(&p.tmO);
    if (p.res != nullptr) tma_prefetch_desc(&p.tmR);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < STAGES; ++s) {
        mbar_init(full_bar(s), 1);
        mbar_init(empty_bar(s), 1);
      }
      for (int a = 0; a < 4; ++a) {
        mbar_init(tfull_bar(a), 1);
        mbar_init(tempty_bar(a), 4);
      }
      for (int w = 0; w < 4 * GROUPS; ++w) mbar_init(res_bar(w), 1);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, TMEM_COLS);
    tmem_relinquish();
  }
  if (warp >= 2) {
    for (int i = threadIdx.x - 64; i < p.cout; i += 128 * GROUPS) s_bias[i] = p.bias[i % p.bias_n];
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      const int mt = tile / p.n_tiles, nt = tile - mt * p.n_tiles;
#pragma unroll 1
      for (int kb = 0; kb < p.num_kb; ++kb) {
        mbar_wait(empty_bar(stage), phase ^ 1u);
        if (elect_one()) {
          const uint32_t st_base = base + stage * STAGE_BYTES;
          mbar_arrive_expect_tx(full_bar(stage), STAGE_BYTES);
          tma_load_2d(st_base, &p.tmA, full_bar(stage), kb * KC, mt * kTileM);
          tma_load_2d(st_base + A_BYTES, &p.tmB, full_bar(stage), kb * KC, nt * NT);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc = make_idesc_f16(kTileM, NT, p.act_bf16);
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const int acc = it & 3;
      const uint32_t acc_phase = (it >> 2) & 1;
      mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * NT;
#pragma unroll 1
      for (int kb = 0; kb < p.num_kb; ++kb) {
        mbar_wait(full_bar(stage), phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t st_base = base + stage * STAGE_BYTES;
          const uint64_t a_desc = make_kmajor_desc(st_base, KCB);
          const uint64_t b_desc = make_kmajor_desc(st_base + A_BYTES, KCB);
#pragma unroll
          for (int k = 0; k < KCB / 32; ++k) umma_f16(d_tmem, a_desc + 2u * k, b_desc + 2u * k, idesc, (kb | k) != 0);
          umma_commit(empty_bar(stage));
          if (kb == p.num_kb - 1) umma_commit(tfull_bar(acc));
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else {
    const int q = warp & 3;
    const int grp = (warp - 2) >> 2;
    const int row_in_tile = q * 32 + lane;
    int it = grp;
    for (int tile = blockIdx.x + grp * gridDim.x; tile < p.num_tiles; tile += GROUPS * gridDim.x, it += GROUPS) {
      const int mt = p.n_tiles == 1 ? tile : tile / p.n_tiles, nt = tile - mt * p.n_tiles;
      const int acc = it & 3;
      const uint32_t acc_phase = (it >> 2) & 1;
      constexpr int BOXC = NT < 64 ? NT : 64;
      constexpr uint32_t BOX_BYTES = 32u * BOXC * 2u;
      const uint32_t stg = staging_base + static_cast<uint32_t>((warp - 2) * (NT / BOXC)) * BOX_BYTES;
      const uint32_t swz = BOXC == 64 ? (lane & 7) : ((lane >> 1) & 3);
      const bool tma_res = pw_tma_out<NT>() && p.res != nullptr;
      if constexpr (pw_tma_out<NT>()) {
        // The staging tile is free once this warp's previous store has read it. With a residual the tile is first
        // FILLED with the residual rows by TMA (same box geometry and swizzle as the store), issued before the wait
        // for the accumulator so its latency hides behind the MMAs; the epilogue then adds in place.
        if (lane == 0) {
          bulk_wait_read<0>();
          if (tma_res) {
            mbar_arrive_expect_tx(res_bar(warp - 2), 32u * NT * 2u);
#pragma unroll
            for (int bx = 0; bx < NT / BOXC; ++bx)
              tma_load_2d(stg + bx * BOX_BYTES, &p.tmR, res_bar(warp - 2), nt * NT + bx * BOXC, mt * kTileM + q * 32);
          }
        }
        __syncwarp();
      }
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
      if (tma_res) mbar_wait(res_bar(warp - 2), ((it - grp) / GROUPS) & 1);
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * NT;
      const long long row = static_cast<long long>(mt) * kTileM + row_in_tile;
      const bool valid = row < p.total_rows;
      const long long off = row * p.cout + nt * NT;
      // Output rows leave through swizzled TMA stores: a thread's 16-byte chunks go to the staging tile at
      // chunk ^ f(row) (the 64B / 128B swizzle patterns), which makes the shared-memory writes conflict free and the
      // global writes whole lines; direct 16-byte stores at a row stride touched 32 half-used sectors per request.
#pragma unroll
      for (int c0 = 0; c0 < NT; c0 += 32) {
        uint32_t r[32];
        tmem_ld32(t_row + c0, r);
        tmem_ld_wait();
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]) + s_bias[nt * NT + c0 + j];
        if (tma_res) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int cc = c0 / 8 + j;
            const uint32_t a = stg + (cc / (BOXC / 8)) * BOX_BYTES + lane * (BOXC * 2) + (((cc % (BOXC / 8)) ^ swz) << 4);
            uint4 rv;
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(rv.x), "=r"(rv.y), "=r"(rv.z), "=r"(rv.w) : "r"(a) : "memory");
            const uint32_t w[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const float2 f = unpack16(w[t], p.act_bf16);
              v[8 * j + 2 * t] += f.x;
              v[8 * j + 2 * t + 1] += f.y;
            }
          }
        } else if (p.res != nullptr && valid) {
          const uint4* rp = reinterpret_cast<const uint4*>(p.res + off + c0);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint4 rv = rp[j];
            const uint32_t w[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const float2 f = unpack16(w[t], p.act_bf16);
              v[8 * j + 2 * t] += f.x;
              v[8 * j + 2 * t + 1] += f.y;
            }
          }
        }
        if (p.relu) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        if constexpr (pw_tma_out<NT>()) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int cc = c0 / 8 + j;                       // 16-byte chunk of the row (compile-time)
            const uint32_t a = stg + (cc / (BOXC / 8)) * BOX_BYTES + lane * (BOXC * 2) + (((cc % (BOXC / 8)) ^ swz) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(pack16(v[8 * j], v[8 * j + 1], p.act_bf16)),
                         "r"(pack16(v[8 * j + 2], v[8 * j + 3], p.act_bf16)), "r"(pack16(v[8 * j + 4], v[8 * j + 5], p.act_bf16)),
                         "r"(pack16(v[8 * j + 6], v[8 * j + 7], p.act_bf16))
                         : "memory");
          }
        } else if (valid) {
          uint4* dst = reinterpret_cast<uint4*>(p.out + off + c0);
#pragma unroll
          for (int j = 0; j < 4; ++j)
            dst[j] = make_uint4(pack16(v[8 * j], v[8 * j + 1], p.act_bf16), pack16(v[8 * j + 2], v[8 * j + 3], p.act_bf16),
                                pack16(v[8 * j + 4], v[8 * j + 5], p.act_bf16), pack16(v[8 * j + 6], v[8 * j + 7], p.act_bf16));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
      if constexpr (pw_tma_out<NT>()) {
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
#pragma unroll
          for (int bx = 0; bx < NT / BOXC; ++bx)
            tma_store_2d(&p.tmO, stg + bx * BOX_BYTES, nt * NT + bx * BOXC, mt * kTileM + q * 32);
          bulk_commit();
        }
      }
    }
  }

  if (warp >= 2 && lane == 0) bulk_wait_all<0>();   // outstanding output stores read shared memory of this CTA
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------------------
// CUDA-core ops on NHWC 16-bit activations
// ------------------------------------------------------------------------------------------------------------
// depthwise k x k conv (pad k/2) + folded BN + optional ReLU; one thread = one output pixel x 8 channels
__global__ void __launch_bounds__(256) dw_conv_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out,
                                                      const float* __restrict__ w /*[k*k][C]*/, const float* __restrict__ bias,
                                                      long long patches, int C, int hin, int hout, int k, int stride, int relu,
                                                      int bf16) {
  const int cg = C >> 3;
  const long long total = patches * hout * hout * cg;
  const int pad = k >> 1;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % cg) * 8;
    long long t = i / cg;
    const int ox = static_cast<int>(t % hout);
    t /= hout;
    const int oy = static_cast<int>(t % hout);
    const long long n = t / hout;
    float acc[8];
    {
      const float4 b0 = *reinterpret_cast<const float4*>(bias + c8);
      const float4 b1 = *reinterpret_cast<const float4*>(bias + c8 + 4);
      acc[0] = b0.x; acc[1] = b0.y; acc[2] = b0.z; acc[3] = b0.w;
      acc[4] = b1.x; acc[5] = b1.y; acc[6] = b1.z; acc[7] = b1.w;
    }
    for (int ky = 0; ky < k; ++ky) {
      const int iy = oy * stride + ky - pad;
      if (iy < 0 || iy >= hin) continue;
      for (int kx = 0; kx < k; ++kx) {
        const int ix = ox * stride + kx - pad;
        if (ix < 0 || ix >= hin) continue;
        const uint4 xv = *reinterpret_cast<const uint4*>(in + ((n * hin + iy) * hin + ix) * C + c8);
        const float* wp = w + (ky * k + kx) * C + c8;
        const float4 w0 = __ldg(reinterpret_cast<const float4*>(wp));
        const float4 w1 = __ldg(reinterpret_cast<const float4*>(wp + 4));
        const float2 x0 = unpack16(xv.x, bf16), x1 = unpack16(xv.y, bf16), x2 = unpack16(xv.z, bf16), x3 = unpack16(xv.w, bf16);
        acc[0] = fmaf(x0.x, w0.x, acc[0]); acc[1] = fmaf(x0.y, w0.y, acc[1]);
        acc[2] = fmaf(x1.x, w0.z, acc[2]); acc[3] = fmaf(x1.y, w0.w, acc[3]);
        acc[4] = fmaf(x2.x, w1.x, acc[4]); acc[5] = fmaf(x2.y, w1.y, acc[5]);
        acc[6] = fmaf(x3.x, w1.z, acc[6]); acc[7] = fmaf(x3.y, w1.w, acc[7]);
      }
    }
    if (relu) {
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = fmaxf(acc[j], 0.f);
    }
    *reinterpret_cast<uint4*>(out + ((n * hout + oy) * hout + ox) * C + c8) =
        make_uint4(pack16(acc[0], acc[1], bf16), pack16(acc[2], acc[3], bf16), pack16(acc[4], acc[5], bf16),
                   pack16(acc[6], acc[7], bf16));
  }
}

// Register-blocked depthwise conv for the shapes the NAS nets use (k in {3, 5}, stride in {1, 2}): a thread owns
// 8 channels x a strip of 4 output pixels of one row. Per ky it loads the K weight vectors once and walks the
// (4 - 1) * S + K input columns once, so an input vector is fetched and unpacked once per row instead of once per
// tap (k = 5, stride 1: 40 loads / 4 outputs instead of 100) and the tap loops are compile-time unrolled.
template <int K, int S>
__global__ void __launch_bounds__(256) dw_conv_strip_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out,
                                                            const float* __restrict__ w /*[k*k][C]*/,
                                                            const float* __restrict__ bias, long long patches, int C, int hin,
                                                            int hout, int relu, int bf16) {
  constexpr int SW = 4;                       // outputs per thread (hout is a multiple of 4 for every NAS stage)
  constexpr int NIN = (SW - 1) * S + K;       // input columns a strip touches
  constexpr int PAD = K >> 1;
  const int cg = C >> 3;
  const int strips = hout / SW;
  const long long total = patches * hout * strips * cg;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % cg) * 8;
    long long t = i / cg;
    const int sx = static_cast<int>(t % strips);
    t /= strips;
    const int oy = static_cast<int>(t % hout);
    const long long n = t / hout;
    // accumulators, inputs and weights are kept as float2 pairs: FFMA2 (fma.rn.f32x2, sm_100) does two FMAs per instruction
    float2 acc[SW][4];
    {
      const float4 b0 = *reinterpret_cast<const float4*>(bias + c8);
      const float4 b1 = *reinterpret_cast<const float4*>(bias + c8 + 4);
#pragma unroll
      for (int j = 0; j < SW; ++j) {
        acc[j][0] = make_float2(b0.x, b0.y); acc[j][1] = make_float2(b0.z, b0.w);
        acc[j][2] = make_float2(b1.x, b1.y); acc[j][3] = make_float2(b1.z, b1.w);
      }
    }
    const int ix0 = sx * SW * S - PAD;
#pragma unroll
    for (int ky = 0; ky < K; ++ky) {
      const int iy = oy * S + ky - PAD;
      if (iy < 0 || iy >= hin) continue;       // warp-uniform: a warp covers one output row
      float2 wk[K][4];
#pragma unroll
      for (int kx = 0; kx < K; ++kx) {
        const float* wp = w + (ky * K + kx) * C + c8;
        const float4 w0 = __ldg(reinterpret_cast<const float4*>(wp));
        const float4 w1 = __ldg(reinterpret_cast<const float4*>(wp + 4));
        wk[kx][0] = make_float2(w0.x, w0.y); wk[kx][1] = make_float2(w0.z, w0.w);
        wk[kx][2] = make_float2(w1.x, w1.y); wk[kx][3] = make_float2(w1.z, w1.w);
      }
      const uint16_t* row = in + ((n * hin + iy) * hin) * C + c8;
#pragma unroll
      for (int c = 0; c < NIN; ++c) {
        const int ix = ix0 + c;
        if (ix < 0 || ix >= hin) continue;
        const uint4 xv = *reinterpret_cast<const uint4*>(row + static_cast<long long>(ix) * C);
        const float2 x[4] = {unpack16(xv.x, bf16), unpack16(xv.y, bf16), unpack16(xv.z, bf16), unpack16(xv.w, bf16)};
#pragma unroll
        for (int j = 0; j < SW; ++j) {
          const int kx = c - j * S;            // compile-time after unrolling
          if (kx >= 0 && kx < K) {
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[j][e] = __ffma2_rn(x[e], wk[kx][e], acc[j][e]);
          }
        }
      }
    }
    uint16_t* orow = out + ((n * hout + oy) * hout + sx * SW) * C + c8;
#pragma unroll
    for (int j = 0; j < SW; ++j) {
      if (relu) {
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[j][e] = make_float2(fmaxf(acc[j][e].x, 0.f), fmaxf(acc[j][e].y, 0.f));
      }
      *reinterpret_cast<uint4*>(orow + static_cast<long long>(j) * C) =
          make_uint4(pack16(acc[j][0].x, acc[j][0].y, bf16), pack16(acc[j][1].x, acc[j][1].y, bf16),
                     pack16(acc[j][2].x, acc[j][2].y, bf16), pack16(acc[j][3].x, acc[j][3].y, bf16));
    }
  }
}

// Depthwise conv through shared memory. A patch's NHWC map is contiguous in HBM, so a unit of G consecutive patches is
// ONE bulk async copy into a two-deep shared-memory ring (the copy of unit u+1 runs under the arithmetic of unit u) and
// every input byte crosses HBM -> L2 -> SM exactly once. A thread owns 8 channels x a VERTICAL strip of SH output rows
// at one output column; consecutive threads walk (channel group, column), so a warp's 16-byte shared loads and its
// 16-byte global stores are contiguous. Per kx the K weight vectors sit in registers and the (SH-1)*S+K input rows are
// loaded once each. Out-of-image taps load a 16-byte zero vector instead (one select on the address) - no divergent
// branches; the activation type is a template parameter so the 16 -> 32 bit unpack is one instruction per value.
template <int K, int S, int SH, bool BF16>
__global__ void __launch_bounds__(256) dw_conv_smem_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out,
                                                           const float* __restrict__ w /*[k*k][C]*/,
                                                           const float* __restrict__ bias, int patches, int C, int hin,
                                                           int hout, int G, int relu) {
  constexpr int bf16 = BF16 ? 1 : 0;
  extern __shared__ __align__(128) uint8_t dw_smem[];
  constexpr int PAD = K >> 1;
  constexpr int NR = (SH - 1) * S + K;         // input rows a strip touches
  const int cg = C >> 3;
  const int map_elems = hin * hin * C;
  const uint32_t unit_bytes = static_cast<uint32_t>(G) * map_elems * 2;
  float* s_w = reinterpret_cast<float*>(dw_smem);                    // [K*K][C] weights, then [C] bias
  const int w_floats = (K * K + 1) * C;
  const uint32_t buf_off = (static_cast<uint32_t>(w_floats) * 4 + 127) & ~127u;
  const uint32_t bar0 = smem_u32(dw_smem + buf_off + 2 * unit_bytes);
  const uint16_t* s_zero = reinterpret_cast<const uint16_t*>(dw_smem + buf_off + 2 * unit_bytes + 16);
  if (threadIdx.x < 4) reinterpret_cast<uint32_t*>(dw_smem + buf_off + 2 * unit_bytes + 16)[threadIdx.x] = 0u;
  for (int i = threadIdx.x; i < K * K * C; i += blockDim.x) s_w[i] = w[i];
  for (int i = threadIdx.x; i < C; i += blockDim.x) s_w[K * K * C + i] = bias[i];
  if (threadIdx.x == 0) {
    mbar_init(bar0, 1);
    mbar_init(bar0 + 8, 1);
    fence_mbar_init();
  }
  __syncthreads();
  const int units = (patches + G - 1) / G;
  auto issue = [&](int u, int slot) {          // one thread: bulk copy of unit u (the tail unit may hold fewer patches)
    const int np = min(G, patches - u * G);
    const uint32_t bytes = static_cast<uint32_t>(np) * map_elems * 2;
    const uint32_t bar = bar0 + 8 * slot;
    mbar_arrive_expect_tx(bar, bytes);
    const uint8_t* src = reinterpret_cast<const uint8_t*>(in) + static_cast<size_t>(u) * unit_bytes;
    const uint32_t dst = smem_u32(dw_smem + buf_off + slot * unit_bytes);
    for (uint32_t o = 0; o < bytes; o += 32768) {
      const uint32_t n = min(32768u, bytes - o);
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst + o),
                   "l"(src + o), "r"(n), "r"(bar)
                   : "memory");
    }
  };
  if (threadIdx.x == 0 && static_cast<int>(blockIdx.x) < units) issue(blockIdx.x, 0);
  const int strips = hout / SH;
  const int items_per_patch = strips * hout * cg;
  int it = 0;
  for (int u = blockIdx.x; u < units; u += gridDim.x, ++it) {
    const int slot = it & 1;
    if (threadIdx.x == 0 && u + static_cast<int>(gridDim.x) < units) issue(u + gridDim.x, slot ^ 1);
    mbar_wait(bar0 + 8 * slot, (it >> 1) & 1);
    const uint16_t* buf = reinterpret_cast<const uint16_t*>(dw_smem + buf_off + slot * unit_bytes);
    const int np = min(G, patches - u * G);
    for (int e = threadIdx.x; e < np * items_per_patch; e += blockDim.x) {
      const int c8 = (e % cg) * 8;
      int t = e / cg;
      const int ox = t % hout;
      t /= hout;
      const int ys = t % strips;
      const int pl = t / strips;
      const uint16_t* map = buf + pl * map_elems + c8;
      float2 acc[SH][4];
      {
        const float4 b0 = *reinterpret_cast<const float4*>(s_w + K * K * C + c8);
        const float4 b1 = *reinterpret_cast<const float4*>(s_w + K * K * C + c8 + 4);
#pragma unroll
        for (int j = 0; j < SH; ++j) {
          acc[j][0] = make_float2(b0.x, b0.y); acc[j][1] = make_float2(b0.z, b0.w);
          acc[j][2] = make_float2(b1.x, b1.y); acc[j][3] = make_float2(b1.z, b1.w);
        }
      }
      const int iy0 = ys * SH * S - PAD;
#pragma unroll
      for (int kx = 0; kx < K; ++kx) {
        const int ix = ox * S + kx - PAD;
        const bool x_ok = ix >= 0 && ix < hin;
        float2 wk[K][4];
#pragma unroll
        for (int ky = 0; ky < K; ++ky) {
          const float* wp = s_w + (ky * K + kx) * C + c8;
          const float4 w0 = *reinterpret_cast<const float4*>(wp);
          const float4 w1 = *reinterpret_cast<const float4*>(wp + 4);
          wk[ky][0] = make_float2(w0.x, w0.y); wk[ky][1] = make_float2(w0.z, w0.w);
          wk[ky][2] = make_float2(w1.x, w1.y); wk[ky][3] = make_float2(w1.z, w1.w);
        }
#pragma unroll
        for (int r = 0; r < NR; ++r) {
          const int iy = iy0 + r;
          const bool ok = x_ok && iy >= 0 && iy < hin;
          const uint4 xv = *reinterpret_cast<const uint4*>(ok ? map + (iy * hin + ix) * C : s_zero);
          const float2 x[4] = {unpack16(xv.x, bf16), unpack16(xv.y, bf16), unpack16(xv.z, bf16), unpack16(xv.w, bf16)};
#pragma unroll
          for (int j = 0; j < SH; ++j) {
            const int ky = r - j * S;          // compile-time after unrolling
            if (ky >= 0 && ky < K) {
#pragma unroll
              for (int q = 0; q < 4; ++q) acc[j][q] = __ffma2_rn(x[q], wk[ky][q], acc[j][q]);
            }
          }
        }
      }
      uint16_t* optr = out + ((static_cast<size_t>(u) * G + pl) * hout + ys * SH) * hout * C + ox * C + c8;
#pragma unroll
      for (int j = 0; j < SH; ++j) {
        if (relu) {
#pragma unroll
          for (int q = 0; q < 4; ++q) acc[j][q] = make_float2(fmaxf(acc[j][q].x, 0.f), fmaxf(acc[j][q].y, 0.f));
        }
        *reinterpret_cast<uint4*>(optr + static_cast<size_t>(j) * hout * C) =
            make_uint4(pack16(acc[j][0].x, acc[j][0].y, bf16), pack16(acc[j][1].x, acc[j][1].y, bf16),
                       pack16(acc[j][2].x, acc[j][2].y, bf16), pack16(acc[j][3].x, acc[j][3].y, bf16));
      }
    }
    __syncthreads();                           // every thread is done with this slot before it is refilled
  }
}

// The same kernel in packed half2 arithmetic for fp16 activations: fp16 weights (converted while they are staged in shared
// memory), fp16 accumulators, no unpacking - HFMA2 issues at twice the FP32 FMA rate and a thread needs 40 instead of ~100
// registers. The 9 / 25-term fp16 accumulation costs ~1e-4 of descriptor error against the 1e-3 gate (CPU emulation of the
// whole net: wang2 8.4e-5 -> 1.5e-4, wang3 1.2e-4 -> 1.8e-4, wang4 1.9e-4 -> 2.2e-4 max-abs); HN_NAS_DW_F32=1 keeps the
// fp32 kernel. bf16 activations always use fp32 arithmetic (8-bit mantissa accumulators would not hold the gate).
template <int K, int S, int SH>
__global__ void __launch_bounds__(256) dw_conv_smem_h2_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out,
                                                              const float* __restrict__ w /*[k*k][C]*/,
                                                              const float* __restrict__ bias, int patches, int C, int hin,
                                                              int hout, int G, int relu) {
  extern __shared__ __align__(128) uint8_t dw_smem[];
  constexpr int PAD = K >> 1;
  constexpr int NR = (SH - 1) * S + K;
  const int cg = C >> 3;
  const int map_elems = hin * hin * C;
  const uint32_t unit_bytes = static_cast<uint32_t>(G) * map_elems * 2;
  __half* s_w = reinterpret_cast<__half*>(dw_smem);                  // [K*K][C] weights, then [C] bias (fp16)
  const int w_halfs = (K * K + 1) * C;
  const uint32_t buf_off = (static_cast<uint32_t>(w_halfs) * 2 + 127) & ~127u;
  const uint32_t bar0 = smem_u32(dw_smem + buf_off + 2 * unit_bytes);
  const uint16_t* s_zero = reinterpret_cast<const uint16_t*>(dw_smem + buf_off + 2 * unit_bytes + 16);
  if (threadIdx.x < 4) reinterpret_cast<uint32_t*>(dw_smem + buf_off + 2 * unit_bytes + 16)[threadIdx.x] = 0u;
  for (int i = threadIdx.x; i < K * K * C; i += blockDim.x) s_w[i] = __float2half_rn(w[i]);
  for (int i = threadIdx.x; i < C; i += blockDim.x) s_w[K * K * C + i] = __float2half_rn(bias[i]);
  if (threadIdx.x == 0) {
    mbar_init(bar0, 1);
    mbar_init(bar0 + 8, 1);
    fence_mbar_init();
  }
  __syncthreads();
  const int units = (patches + G - 1) / G;
  auto issue = [&](int u, int slot) {
    const int np = min(G, patches - u * G);
    const uint32_t bytes = static_cast<uint32_t>(np) * map_elems * 2;
    const uint32_t bar = bar0 + 8 * slot;
    mbar_arrive_expect_tx(bar, bytes);
    const uint8_t* src = reinterpret_cast<const uint8_t*>(in) + static_cast<size_t>(u) * unit_bytes;
    const uint32_t dst = smem_u32(dw_smem + buf_off + slot * unit_bytes);
    for (uint32_t o = 0; o < bytes; o += 32768) {
      const uint32_t n = min(32768u, bytes - o);
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst + o),
                   "l"(src + o), "r"(n), "r"(bar)
                   : "memory");
    }
  };
  if (threadIdx.x == 0 && static_cast<int>(blockIdx.x) < units) issue(blockIdx.x, 0);
  const int strips = hout / SH;
  const int items_per_patch = strips * hout * cg;
  const __half2 hzero = __float2half2_rn(0.f);
  int it = 0;
  for (int u = blockIdx.x; u < units; u += gridDim.x, ++it) {
    const int slot = it & 1;
    if (threadIdx.x == 0 && u + static_cast<int>(gridDim.x) < units) issue(u + gridDim.x, slot ^ 1);
    mbar_wait(bar0 + 8 * slot, (it >> 1) & 1);
    const uint16_t* buf = reinterpret_cast<const uint16_t*>(dw_smem + buf_off + slot * unit_bytes);
    const int np = min(G, patches - u * G);
    for (int e = threadIdx.x; e < np * items_per_patch; e += blockDim.x) {
      const int c8 = (e % cg) * 8;
      int t = e / cg;
      const int ox = t % hout;
      t /= hout;
      const int ys = t % strips;
      const int pl = t / strips;
      const uint16_t* map = buf + pl * map_elems + c8;
      __half2 acc[SH][4];
      {
        const uint4 b = *reinterpret_cast<const uint4*>(s_w + K * K * C + c8);
#pragma unroll
        for (int j = 0; j < SH; ++j) {
          acc[j][0] = *reinterpret_cast<const __half2*>(&b.x); acc[j][1] = *reinterpret_cast<const __half2*>(&b.y);
          acc[j][2] = *reinterpret_cast<const __half2*>(&b.z); acc[j][3] = *reinterpret_cast<const __half2*>(&b.w);
        }
      }
      const int iy0 = ys * SH * S - PAD;
#pragma unroll
      for (int kx = 0; kx < K; ++kx) {
        const int ix = ox * S + kx - PAD;
        const bool x_ok = ix >= 0 && ix < hin;
        uint4 wk[K];
#pragma unroll
        for (int ky = 0; ky < K; ++ky) wk[ky] = *reinterpret_cast<const uint4*>(s_w + (ky * K + kx) * C + c8);
#pragma unroll
        for (int r = 0; r < NR; ++r) {
          const int iy = iy0 + r;
          const bool ok = x_ok && iy >= 0 && iy < hin;
          const uint4 xv = *reinterpret_cast<const uint4*>(ok ? map + (iy * hin + ix) * C : s_zero);
          const __half2 x[4] = {*reinterpret_cast<const __half2*>(&xv.x), *reinterpret_cast<const __half2*>(&xv.y),
                                *reinterpret_cast<const __half2*>(&xv.z), *reinterpret_cast<const __half2*>(&xv.w)};
#pragma unroll
          for (int j = 0; j < SH; ++j) {
            const int ky = r - j * S;          // compile-time after unrolling
            if (ky >= 0 && ky < K) {
              const __half2 wv[4] = {*reinterpret_cast<const __half2*>(&wk[ky].x), *reinterpret_cast<const __half2*>(&wk[ky].y),
                                     *reinterpret_cast<const __half2*>(&wk[ky].z), *reinterpret_cast<const __half2*>(&wk[ky].w)};
#pragma unroll
              for (int q = 0; q < 4; ++q) acc[j][q] = __hfma2(x[q], wv[q], acc[j][q]);
            }
          }
        }
      }
      uint16_t* optr = out + ((static_cast<size_t>(u) * G + pl) * hout + ys * SH) * hout * C + ox * C + c8;
#pragma unroll
      for (int j = 0; j < SH; ++j) {
        if (relu) {
#pragma unroll
          for (int q = 0; q < 4; ++q) acc[j][q] = __hmax2(acc[j][q], hzero);
        }
        *reinterpret_cast<uint4*>(optr + static_cast<size_t>(j) * hout * C) =
            make_uint4(*reinterpret_cast<const uint32_t*>(&acc[j][0]), *reinterpret_cast<const uint32_t*>(&acc[j][1]),
                       *reinterpret_cast<const uint32_t*>(&acc[j][2]), *reinterpret_cast<const uint32_t*>(&acc[j][3]));
      }
    }
    __syncthreads();                           // every thread is done with this slot before it is refilled
  }
}

// MaxPool2d(3, stride 2, padding 1) through the same bulk-copied shared-memory ring as the depthwise kernel: a thread
// owns 8 channels x a vertical strip of 4 output rows and takes packed 16-bit maxima directly (max is exact in fp16 /
// bf16, NaNs propagate like torch); out-of-image taps read a -inf vector.
template <bool BF16>
__global__ void __launch_bounds__(256) maxpool_smem_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out,
                                                           int patches, int C, int hin, int hout, int G) {
  extern __shared__ __align__(128) uint8_t dw_smem[];
  constexpr int SH = 4, NR = (SH - 1) * 2 + 3;
  const int cg = C >> 3;
  const int map_elems = hin * hin * C;
  const uint32_t unit_bytes = static_cast<uint32_t>(G) * map_elems * 2;
  const uint32_t bar0 = smem_u32(dw_smem + 2 * unit_bytes);
  const uint32_t ninf = BF16 ? 0xFF80FF80u : 0xFC00FC00u;
  const uint16_t* s_ninf = reinterpret_cast<const uint16_t*>(dw_smem + 2 * unit_bytes + 16);
  if (threadIdx.x < 4) reinterpret_cast<uint32_t*>(dw_smem + 2 * unit_bytes + 16)[threadIdx.x] = ninf;
  if (threadIdx.x == 0) {
    mbar_init(bar0, 1);
    mbar_init(bar0 + 8, 1);
    fence_mbar_init();
  }
  __syncthreads();
  const int units = (patches + G - 1) / G;
  auto issue = [&](int u, int slot) {
    const int np = min(G, patches - u * G);
    const uint32_t bytes = static_cast<uint32_t>(np) * map_elems * 2;
    const uint32_t bar = bar0 + 8 * slot;
    mbar_arrive_expect_tx(bar, bytes);
    const uint8_t* src = reinterpret_cast<const uint8_t*>(in) + static_cast<size_t>(u) * unit_bytes;
    const uint32_t dst = smem_u32(dw_smem + slot * unit_bytes);
    for (uint32_t o = 0; o < bytes; o += 32768) {
      const uint32_t n = min(32768u, bytes - o);
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst + o),
                   "l"(src + o), "r"(n), "r"(bar)
                   : "memory");
    }
  };
  auto vmax = [](uint32_t a, uint32_t b) -> uint32_t {
    if constexpr (BF16) {
      const __nv_bfloat162 r = __hmax2_nan(*reinterpret_cast<const __nv_bfloat162*>(&a), *reinterpret_cast<const __nv_bfloat162*>(&b));
      return *reinterpret_cast<const uint32_t*>(&r);
    } else {
      const __half2 r = __hmax2_nan(*reinterpret_cast<const __half2*>(&a), *reinterpret_cast<const __half2*>(&b));
      return *reinterpret_cast<const uint32_t*>(&r);
    }
  };
  if (threadIdx.x == 0 && static_cast<int>(blockIdx.x) < units) issue(blockIdx.x, 0);
  const int strips = hout / SH;
  const int items_per_patch = strips * hout * cg;
  int it = 0;
  for (int u = blockIdx.x; u < units; u += gridDim.x, ++it) {
    const int slot = it & 1;
    if (threadIdx.x == 0 && u + static_cast<int>(gridDim.x) < units) issue(u + gridDim.x, slot ^ 1);
    mbar_wait(bar0 + 8 * slot, (it >> 1) & 1);
    const uint16_t* buf = reinterpret_cast<const uint16_t*>(dw_smem + slot * unit_bytes);
    const int np = min(G, patches - u * G);
    for (int e = threadIdx.x; e < np * items_per_patch; e += blockDim.x) {
      const int c8 = (e % cg) * 8;
      int t = e / cg;
      const int ox = t % hout;
      t /= hout;
      const int ys = t % strips;
      const int pl = t / strips;
      const uint16_t* map = buf + pl * map_elems + c8;
      uint4 acc[SH];
#pragma unroll
      for (int j = 0; j < SH; ++j) acc[j] = make_uint4(ninf, ninf, ninf, ninf);
      const int iy0 = ys * SH * 2 - 1;
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int ix = ox * 2 + kx - 1;
        const bool x_ok = ix >= 0 && ix < hin;
#pragma unroll
        for (int r = 0; r < NR; ++r) {
          const int iy = iy0 + r;
          const bool ok = x_ok && iy >= 0 && iy < hin;
          const uint4 xv = *reinterpret_cast<const uint4*>(ok ? map + (iy * hin + ix) * C : s_ninf);
#pragma unroll
          for (int j = 0; j < SH; ++j) {
            const int ky = r - j * 2;          // compile-time after unrolling
            if (ky >= 0 && ky < 3)
              acc[j] = make_uint4(vmax(acc[j].x, xv.x), vmax(acc[j].y, xv.y), vmax(acc[j].z, xv.z), vmax(acc[j].w, xv.w));
          }
        }
      }
      uint16_t* optr = out + ((static_cast<size_t>(u) * G + pl) * hout + ys * SH) * hout * C + ox * C + c8;
#pragma unroll
      for (int j = 0; j < SH; ++j) *reinterpret_cast<uint4*>(optr + static_cast<size_t>(j) * hout * C) = acc[j];
    }
    __syncthreads();
  }
}

// MaxPool2d(kernel 3, stride 2, padding 1): padding never wins (implicit -inf), like torch
__global__ void __launch_bounds__(256) maxpool_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out,
                                                      long long patches, int C, int hin, int hout, int bf16) {
  const int cg = C >> 3;
  const long long total = patches * hout * hout * cg;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % cg) * 8;
    long long t = i / cg;
    const int ox = static_cast<int>(t % hout);
    t /= hout;
    const int oy = static_cast<int>(t % hout);
    const long long n = t / hout;
    float m[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) m[j] = -__int_as_float(0x7f800000);
    for (int ky = 0; ky < 3; ++ky) {
      const int iy = oy * 2 + ky - 1;
      if (iy < 0 || iy >= hin) continue;
      for (int kx = 0; kx < 3; ++kx) {
        const int ix = ox * 2 + kx - 1;
        if (ix < 0 || ix >= hin) continue;
        const uint4 xv = *reinterpret_cast<const uint4*>(in + ((n * hin + iy) * hin + ix) * C + c8);
        const uint32_t wv[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = unpack16(wv[j], bf16);
          m[2 * j] = fmaxf(m[2 * j], f.x);
          m[2 * j + 1] = fmaxf(m[2 * j + 1], f.y);
        }
      }
    }
    *reinterpret_cast<uint4*>(out + ((n * hout + oy) * hout + ox) * C + c8) =
        make_uint4(pack16(m[0], m[1], bf16), pack16(m[2], m[3], bf16), pack16(m[4], m[5], bf16), pack16(m[6], m[7], bf16));
  }
}

// Squeeze-and-excite, in place; one CTA per patch. fc weights fp32: w1 [mid][C], w2 [C][mid].
__global__ void __launch_bounds__(256) se_kernel(uint16_t* __restrict__ x, long long patches, int C, int h, int mid,
                                                 const float* __restrict__ w1, const float* __restrict__ b1,
                                                 const float* __restrict__ w2, const float* __restrict__ b2, int bf16) {
  __shared__ float s_mean[512];
  __shared__ float s_hid[128];
  __shared__ float s_gate[512];
  const int pix = h * h;
  for (long long n = blockIdx.x; n < patches; n += gridDim.x) {
    uint16_t* xp = x + n * pix * C;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      float s = 0.f;
      for (int i = 0; i < pix; ++i) {
        const uint16_t raw = xp[i * C + c];
        s += bf16 ? __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(&raw)) : __half2float(*reinterpret_cast<const __half*>(&raw));
      }
      s_mean[c] = s / static_cast<float>(pix);
    }
    __syncthreads();
    for (int j = threadIdx.x; j < mid; j += blockDim.x) {
      float s = b1[j];
      for (int c = 0; c < C; ++c) s = fmaf(w1[j * C + c], s_mean[c], s);
      s_hid[j] = fmaxf(s, 0.f);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      float s = b2[c];
      for (int j = 0; j < mid; ++j) s = fmaf(w2[c * mid + j], s_hid[j], s);
      s_gate[c] = 1.0f / (1.0f + expf(-s));
    }
    __syncthreads();
    for (int i = threadIdx.x; i < pix * C / 2; i += blockDim.x) {
      uint32_t* p2 = reinterpret_cast<uint32_t*>(xp) + i;
      const int c = (i * 2) % C;
      const float2 f = unpack16(*p2, bf16);
      *p2 = pack16(f.x * s_gate[c], f.y * s_gate[c + 1], bf16);
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
// A run of consecutive ops behind the front stage executed by ONE launch of nas_tail_kernel (nas_tail.cuh), a warpgroup per patch.
struct NasTail {
  int first = 0, last = 0;   // op range [first, last]
  int last_orig = 0;         // packed op whose output the run's last op produces
  int nwg = 0;               // warpgroups (= patches in flight) per CTA
  size_t smem = 0;
  std::vector<int> dst_off;  // per op of the run: byte offset of its output inside a warpgroup's region
  std::vector<int> src_r, res_r, dst_r;   // per op: regions of its inputs / output
  std::vector<int> out_c, out_h, is_pw;   // per op: output channels / side, pointwise?
  TailParams params;
  uint8_t* blob = nullptr;   // device copy of the weight image
};

struct NasState {
  std::vector<NasTail> tails;        // plain form of the ops behind the front stage (op k of the form = packed op tail_first + k):
                                     // activation dumps, and the forward when the folded form is unavailable
  std::vector<int> tail_of_op;       // packed op -> index into tails, or -1
  int tail_first = 0;
  int head_planar = 0;               // the last plain tail launch writes the head GEMM's rows channel-planar (head weight K order permuted)
  std::vector<NasTail> ftails;       // folded form (linear 1x1 convs folded into their consumers): the forward's launches
  uint16_t* headf_w = nullptr;       // folded head: [128][headf_k] 16-bit, channel-planar K order
  float* headf_b = nullptr;
  int headf_k = 0;
  TcParams headf;
  std::vector<hn_nas_op> ops;
  std::vector<PwParams> pw;          // one per op (valid for OP_PW)
  std::vector<size_t> w16_off;       // 16-bit weight offset per op (PW / HEAD)
  float* params = nullptr;           // fp32 blob on the device
  uint16_t* w16 = nullptr;
  uint16_t* slot[3] = {nullptr, nullptr, nullptr};
  uint16_t* head_in = nullptr;       // [head_rows, head_k]
  uint16_t* front_img = nullptr;     // op 1 as a fused-front weight image when stem + op 1 run as one kernel, else null
  CUtensorMap front_tm;              // its output ([chunk * 1024, 32] as 32 x 32 store boxes, 64B swizzle)
  float front_bias2[32];             // op 1's folded BN shift (host copy: a by-value kernel parameter)
  int front_ops = 0;                 // ops the front kernel covers: 2 = stem + pointwise, 1 = stem alone (identity pointwise)
  int front_fdw = 0;                 // != 0: op `front_ops` (depthwise 3 | 5 stride 2, or max-pool = 1) also runs inside the front kernel
  size_t slot_elems = 0;             // per patch
  int chunk = 0;                     // patches per pass (<= handle chunk, capped so the three slots stay <= 4 GiB)
  int head_k = 0;
  int act_bf16 = 0;
  TcParams head;
};

void nas_state_free(NasState* s) {
  if (!s) return;
  cudaFree(s->params);
  cudaFree(s->w16);
  for (auto* p : s->slot) cudaFree(p);
  cudaFree(s->head_in);
  cudaFree(s->front_img);
  for (auto& tl : s->tails) cudaFree(tl.blob);
  for (auto& tl : s->ftails) cudaFree(tl.blob);
  cudaFree(s->headf_w);
  cudaFree(s->headf_b);
  delete s;
}

static uint16_t f2h16(float v, int bf16) {
  if (bf16) {
    __nv_bfloat16 h = __float2bfloat16_rn(v);
    return *reinterpret_cast<uint16_t*>(&h);
  }
  __half h = __float2half_rn(v);
  return *reinterpret_cast<uint16_t*>(&h);
}

static int pick_nt(int cout) {
  if (cout <= 128) return cout;
  if (cout % 128 == 0) return 128;
  if (cout % 96 == 0) return 96;
  if (cout % 64 == 0) return 64;
  return 32;
}

template <int NT, int KCB>
static int launch_pw_cfg(const PwParams& p, int sm_count, cudaStream_t s) {
  auto kern = pw_gemm_kernel<NT, KCB>;
  constexpr size_t smem = pw_smem_bytes<NT, KCB>();
  static DeviceOnce attr_once;
  if (attr_once.first_time()) {
    HN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  }
  if (p.num_tiles <= 0) return HN_OK;
  kern<<<std::min(p.num_tiles, sm_count), pw_threads<NT>(), smem, s>>>(p);
  HN_CUDA(cudaGetLastError());
  count_launch();
  return HN_OK;
}

static int launch_pw(const PwParams& p, int nt, int kcb, int sm_count, cudaStream_t s) {
#define HN_PW_CASE(NT_)                                                    \
  if (nt == NT_) return kcb == 64 ? launch_pw_cfg<NT_, 64>(p, sm_count, s) : launch_pw_cfg<NT_, 128>(p, sm_count, s);
  HN_PW_CASE(32)
  HN_PW_CASE(64)
  HN_PW_CASE(96)
  HN_PW_CASE(128)
#undef HN_PW_CASE
  set_error("pointwise conv: unsupported output tile width %d", nt);
  return HN_ERR_UNSUPPORTED;
}

}  // namespace hn


namespace hn {

// ------------------------------------------------------------------------------------------------------------
// warpgroup-per-patch tail launches (nas_tail.cuh)
// ------------------------------------------------------------------------------------------------------------
static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// The ops behind the front stage as a small SSA program over tensor ids (tensor 0 = the front stage's output). Two forms:
//   plain   one TOp per packed op, a block's residual as an identity second input (activation dumps run this form, so every
//           packed op's output can still be inspected), and
//   folded  every LINEAR 1x1 conv (the `pwl` of an IRFBlock, fbnet_builder.py:455-570: conv + BN, no ReLU) is folded into its
//           consumers: y = relu(W2 (W1 a + b1 + x) + b2) = relu((W2 W1) a + W2 x + (W2 b1 + b2)) is ONE pointwise op with two
//           inputs, and the head conv of model_supernet.py:64-68 absorbs the last block's `pwl`. wang2: 13 ops -> 8 (4 pointwise
//           + 4 depthwise), head K 2048 -> 1024. Products are formed in double precision and rounded once to fp16, so the
//           folded net drops roundings of intermediate activations rather than adding any.
struct TOp {
  int kind = 0;                 // OP_PW / OP_DW / OP_MAXPOOL
  int cin = 0, cout = 0, kernel = 1, stride = 1, hin = 0, hout = 0, relu = 0;
  int in0 = -1, in1 = -1, out = -1;   // tensor ids (in1: second input of a pointwise op)
  int c1 = 0;                   // channels of in1
  int ident1 = 0;               // in1 is added as it is (identity weights)
  std::vector<float> w, w1, b;  // PW: [cout][cin], [cout][c1] (unless ident1), [cout]; DW: [k * k][C], [C]
  int orig = -1;                // packed op whose output this op produces
};

struct TProg {
  std::vector<TOp> ops;
  std::vector<std::pair<int, int>> tensors;   // (channels, side)
  // head: [128][pix * C] in NHWC K order (pixel * C + c) over tensor `head_in`
  int head_in = -1, head_c = 0, head_pix = 0;
  std::vector<float> head_w, head_b;
  bool folded = false;
};

static int tail_pw_shape(int cin, int c1w /*weighted second input channels, 0 = none / identity*/, int cout, int rows) {
  struct S { int cin, c1, cout, rows; };
  static const S table[] = {{32, 0, 32, 256}, {32, 0, 64, 64}, {64, 0, 64, 64}, {64, 0, 128, 16}, {128, 0, 128, 16},
                            {32, 32, 32, 256}, {64, 32, 64, 64}, {64, 64, 64, 64}, {128, 64, 128, 16}};
  for (int i = 0; i < static_cast<int>(sizeof(table) / sizeof(table[0])); ++i)
    if (table[i].cin == cin && table[i].c1 == c1w && table[i].cout == cout && table[i].rows == rows) return i;
  return -1;
}
static int tail_dw_shape(int c, int hin, int hout, int stride) {
  if (hout * stride != hin) return -1;
  if (c == 32 && hout == 16 && stride == 1) return 0;
  if (c == 32 && hout == 8 && stride == 2) return 1;
  if (c == 64 && hout == 8 && stride == 1) return 2;
  if (c == 64 && hout == 4 && stride == 2) return 3;
  if (c == 128 && hout == 4 && stride == 1) return 4;
  return -1;
}
static int tail_op_shape(const TOp& o) {
  switch (o.kind) {
    case OP_PW: return (o.in1 >= 0 && o.ident1 && o.c1 != o.cout) ? -1 : tail_pw_shape(o.cin, (o.in1 >= 0 && !o.ident1) ? o.c1 : 0, o.cout, o.hin * o.hin);
    case OP_DW: return (o.kernel == 3 || o.kernel == 5) ? tail_dw_shape(o.cin, o.hin, o.hout, o.stride) : -1;
    case OP_MAXPOOL: { const int sh = tail_dw_shape(o.cin, o.hin, o.hout, o.stride); return (sh == 1 || sh == 3) ? sh : -1; }
    default: return -1;
  }
}

static int ilog2(int v) { int l = 0; while ((1 << l) < v) ++l; return l; }

// plain form: one TOp per packed op of [first, n_ops - 2]; false if the program does not have the expected structure
static bool tail_prog_plain(const std::vector<hn_nas_op>& ops, const float* params, int first, TProg& pr) {
  const int n_ops = static_cast<int>(ops.size());
  int slot_t[3] = {-1, -1, -1};
  const hn_nas_op& of = ops[first];
  pr.tensors.emplace_back(of.cin, of.hin);
  slot_t[of.src] = 0;
  for (int i = first; i <= n_ops - 2; ++i) {
    const hn_nas_op& o = ops[i];
    if (o.kind != OP_PW && o.kind != OP_DW && o.kind != OP_MAXPOOL) return false;
    TOp t;
    t.kind = o.kind; t.cin = o.cin; t.cout = o.cout; t.kernel = o.kernel; t.stride = o.kind == OP_PW ? 1 : o.stride;
    t.hin = o.hin; t.hout = o.hout; t.relu = o.relu; t.orig = i;
    t.in0 = slot_t[o.src];
    if (t.in0 < 0) return false;
    if (o.kind == OP_PW && o.res >= 0) {
      t.in1 = slot_t[o.res];
      if (t.in1 < 0) return false;
      t.c1 = o.cout; t.ident1 = 1;
    }
    if (o.kind == OP_PW) {
      t.w.assign(params + o.w_off, params + o.w_off + static_cast<size_t>(o.cin) * o.cout);
      t.b.assign(params + o.b_off, params + o.b_off + o.cout);
    } else if (o.kind == OP_DW) {
      t.w.assign(params + o.w_off, params + o.w_off + static_cast<size_t>(o.kernel) * o.kernel * o.cin);
      t.b.assign(params + o.b_off, params + o.b_off + o.cin);
    }
    t.out = static_cast<int>(pr.tensors.size());
    pr.tensors.emplace_back(o.cout, o.hout);
    slot_t[o.dst] = t.out;
    pr.ops.push_back(std::move(t));
  }
  const hn_nas_op& oh = ops[n_ops - 1];
  pr.head_in = slot_t[oh.src];
  if (pr.head_in < 0) return false;
  pr.head_c = oh.cin; pr.head_pix = oh.kernel * oh.kernel;
  const size_t K = static_cast<size_t>(pr.head_pix) * pr.head_c;
  pr.head_w.assign(params + oh.w_off, params + oh.w_off + 128 * K);
  pr.head_b.assign(params + oh.b_off, params + oh.b_off + 128);
  return true;
}

// folded form (see above); false if a value would need more than two inputs in a way the pass does not resolve
static bool tail_prog_folded(const std::vector<hn_nas_op>& ops, const float* params, int first, TProg& pr) {
  struct Term { int t, ct; std::vector<double> M; };                  // M: [C][ct]
  struct Val { bool mat = false; int t = -1, C = 0, H = 0; std::vector<Term> terms; std::vector<double> c; bool set = false; };
  const int n_ops = static_cast<int>(ops.size());
  Val vals[3];
  const hn_nas_op& of = ops[first];
  pr.tensors.emplace_back(of.cin, of.hin);
  vals[of.src].mat = true; vals[of.src].t = 0; vals[of.src].C = of.cin; vals[of.src].H = of.hin; vals[of.src].set = true;
  auto is_identity = [](const Term& tm, int C) {
    if (tm.ct != C) return false;
    for (int r = 0; r < C; ++r)
      for (int k = 0; k < C; ++k)
        if (tm.M[static_cast<size_t>(r) * C + k] != (r == k ? 1.0 : 0.0)) return false;
    return true;
  };
  // emits the pointwise op that computes a linear value (1 or 2 terms) and turns it into a materialised tensor
  auto materialize = [&](Val& v, int relu, int orig) -> bool {
    if (v.mat) return true;
    if (v.terms.empty() || v.terms.size() > 2) return false;
    if (v.terms.size() == 2 && is_identity(v.terms[0], v.C) && !is_identity(v.terms[1], v.C)) std::swap(v.terms[0], v.terms[1]);
    TOp t;
    t.kind = OP_PW; t.cin = v.terms[0].ct; t.cout = v.C; t.hin = t.hout = v.H; t.relu = relu; t.orig = orig;
    t.in0 = v.terms[0].t;
    t.w.assign(v.terms[0].M.begin(), v.terms[0].M.end());
    if (v.terms.size() == 2) {
      t.in1 = v.terms[1].t; t.c1 = v.terms[1].ct;
      t.ident1 = is_identity(v.terms[1], v.C) ? 1 : 0;
      if (!t.ident1) t.w1.assign(v.terms[1].M.begin(), v.terms[1].M.end());
    }
    t.b.assign(v.c.begin(), v.c.end());
    t.out = static_cast<int>(pr.tensors.size());
    pr.tensors.emplace_back(v.C, v.H);
    pr.ops.push_back(std::move(t));
    v.mat = true; v.t = pr.ops.back().out; v.terms.clear(); v.c.clear();
    return true;
  };
  // terms of W * v (v materialised: one term; v linear: W composed with each of its terms), bias W * c
  auto apply = [&](const std::vector<double>& W, int cout, const Val& v, std::vector<Term>& terms, std::vector<double>& bias) {
    if (v.mat) {
      terms.push_back({v.t, v.C, W});
      return;
    }
    for (const Term& tm : v.terms) {
      Term nt{tm.t, tm.ct, std::vector<double>(static_cast<size_t>(cout) * tm.ct, 0.0)};
      for (int r = 0; r < cout; ++r)
        for (int k = 0; k < v.C; ++k) {
          const double wv = W[static_cast<size_t>(r) * v.C + k];
          if (wv == 0.0) continue;
          for (int j = 0; j < tm.ct; ++j) nt.M[static_cast<size_t>(r) * tm.ct + j] += wv * tm.M[static_cast<size_t>(k) * tm.ct + j];
        }
      terms.push_back(std::move(nt));
    }
    for (int r = 0; r < cout; ++r)
      for (int k = 0; k < v.C; ++k) bias[r] += W[static_cast<size_t>(r) * v.C + k] * v.c[k];
  };
  auto add_terms = [&](std::vector<Term>& terms, const Term& tm) {
    for (Term& e : terms)
      if (e.t == tm.t) {
        for (size_t j = 0; j < e.M.size(); ++j) e.M[j] += tm.M[j];
        return;
      }
    terms.push_back(tm);
  };
  for (int i = first; i <= n_ops - 2; ++i) {
    const hn_nas_op& o = ops[i];
    if (!vals[o.src].set) return false;
    if (o.kind == OP_PW) {
      if (o.res >= 0 && !vals[o.res].set) return false;
      for (int attempt = 0; attempt < 3; ++attempt) {
        std::vector<double> W(params + o.w_off, params + o.w_off + static_cast<size_t>(o.cin) * o.cout);
        std::vector<Term> terms;
        std::vector<double> bias(params + o.b_off, params + o.b_off + o.cout);
        apply(W, o.cout, vals[o.src], terms, bias);
        if (o.res >= 0) {
          const Val& rv = vals[o.res];
          if (rv.mat) {
            Term id{rv.t, rv.C, std::vector<double>(static_cast<size_t>(rv.C) * rv.C, 0.0)};
            for (int r = 0; r < rv.C; ++r) id.M[static_cast<size_t>(r) * rv.C + r] = 1.0;
            add_terms(terms, id);
          } else {
            for (const Term& tm : rv.terms) add_terms(terms, tm);
            for (int r = 0; r < o.cout; ++r) bias[r] += rv.c[r];
          }
        }
        if (terms.size() > 2) {     // too many inputs: compute a linear operand for real first, then try again
          if (!vals[o.src].mat) { if (!materialize(vals[o.src], 0, -1)) return false; }
          else if (o.res >= 0 && !vals[o.res].mat) { if (!materialize(vals[o.res], 0, -1)) return false; }
          else return false;
          continue;
        }
        Val out;
        out.C = o.cout; out.H = o.hin; out.terms = std::move(terms); out.c = std::move(bias); out.set = true;
        if (o.relu && !materialize(out, 1, i)) return false;
        vals[o.dst] = std::move(out);
        break;
      }
      if (!vals[o.dst].set) return false;
    } else if (o.kind == OP_DW || o.kind == OP_MAXPOOL) {
      if (!materialize(vals[o.src], 0, -1)) return false;
      TOp t;
      t.kind = o.kind; t.cin = o.cin; t.cout = o.cout; t.kernel = o.kernel; t.stride = o.stride; t.hin = o.hin; t.hout = o.hout; t.relu = o.relu;
      t.orig = i; t.in0 = vals[o.src].t;
      if (o.kind == OP_DW) {
        t.w.assign(params + o.w_off, params + o.w_off + static_cast<size_t>(o.kernel) * o.kernel * o.cin);
        t.b.assign(params + o.b_off, params + o.b_off + o.cin);
      }
      t.out = static_cast<int>(pr.tensors.size());
      pr.tensors.emplace_back(o.cout, o.hout);
      pr.ops.push_back(std::move(t));
      Val out;
      out.mat = true; out.t = pr.ops.back().out; out.C = o.cout; out.H = o.hout; out.set = true;
      vals[o.dst] = std::move(out);
    } else {
      return false;
    }
  }
  // head conv: absorbs a linear value with ONE source tensor
  const hn_nas_op& oh = ops[n_ops - 1];
  Val& hv = vals[oh.src];
  if (!hv.set) return false;
  const int pix = oh.kernel * oh.kernel, C = oh.cin;
  const float* Wh = params + oh.w_off;           // [128][pix * C]
  pr.head_pix = pix;
  pr.head_b.assign(params + oh.b_off, params + oh.b_off + 128);
  if (!hv.mat && hv.terms.size() == 1 && hv.terms[0].ct % 8 == 0 && (pix * hv.terms[0].ct) % 128 == 0) {
    const Term& tm = hv.terms[0];
    pr.head_in = tm.t; pr.head_c = tm.ct;
    pr.head_w.assign(static_cast<size_t>(128) * pix * tm.ct, 0.f);
    std::vector<double> acc(tm.ct);
    for (int o2 = 0; o2 < 128; ++o2) {
      double bsum = pr.head_b[o2];
      for (int px = 0; px < pix; ++px) {
        std::fill(acc.begin(), acc.end(), 0.0);
        const float* wrow = Wh + (static_cast<size_t>(o2) * pix + px) * C;
        for (int c = 0; c < C; ++c) {
          const double wv = wrow[c];
          bsum += wv * hv.c[c];
          for (int j = 0; j < tm.ct; ++j) acc[j] += wv * tm.M[static_cast<size_t>(c) * tm.ct + j];
        }
        for (int j = 0; j < tm.ct; ++j) pr.head_w[(static_cast<size_t>(o2) * pix + px) * tm.ct + j] = static_cast<float>(acc[j]);
      }
      pr.head_b[o2] = static_cast<float>(bsum);
    }
  } else {
    if (!materialize(hv, 0, n_ops - 2)) return false;
    pr.head_in = hv.t; pr.head_c = C;
    pr.head_w.assign(Wh, Wh + static_cast<size_t>(128) * pix * C);
  }
  pr.folded = true;
  return true;
}

// Finalises tail launch [first, last] of `pr`: region offsets, warpgroups per CTA, weight image on the device.
static int tail_build(hn_handle* h, const TProg& pr, int first, int last, int launch_id, NasTail& tl) {
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t r = off; off = align_up(off + bytes, 128); return r; };
  const int n = last - first + 1;
  if (n > kTailMaxOps) return HN_ERR_UNSUPPORTED;
  std::vector<size_t> w_off(n, 0), b_off(n, 0);
  // constant tiles: "ones" A tile (K plane 0: columns 0, 1 = 1.0; K plane 1 = 2 KB of zeros, also the depthwise zero padding),
  // 128 bytes of -inf (max-pool padding), 16 x 16 identity B tile
  const size_t ones_off = take(4096 + 128);
  const size_t eye_off = take(512);
  size_t region_bytes = 0;
  bool big_map = false;
  auto wc1 = [](const TOp& o) { return (o.in1 >= 0 && !o.ident1) ? o.c1 : 0; };   // weighted second-input channels
  for (int i = first; i <= last; ++i) {
    const TOp& o = pr.ops[i];
    if (tail_op_shape(o) < 0) return HN_ERR_UNSUPPORTED;
    // weights and biases are stored as fp16 (the bias as hi + lo): values outside its range keep the per-op path (fp32 biases)
    auto fits16 = [](const std::vector<float>& v) {
      for (float x : v)
        if (!(std::fabs(x) < 60000.f)) return false;
      return true;
    };
    if (!fits16(o.w) || !fits16(o.w1) || !fits16(o.b)) return HN_ERR_UNSUPPORTED;
    const size_t in_b = static_cast<size_t>(o.cin) * o.hin * o.hin * 2, out_b = static_cast<size_t>(o.cout) * o.hout * o.hout * 2;
    region_bytes = std::max(region_bytes, std::max(in_b, out_b));
    if (o.in1 >= 0) region_bytes = std::max(region_bytes, static_cast<size_t>(o.c1) * o.hin * o.hin * 2);
    big_map = big_map || o.hin == 16;
    const int k = i - first;
    if (o.kind == OP_PW) w_off[k] = take(static_cast<size_t>(o.cin + 16 + wc1(o)) * o.cout * 2);   // + 16 K columns: bias as fp16 hi + lo
    if (o.kind == OP_DW) { w_off[k] = take(static_cast<size_t>(o.kernel) * o.kernel * o.cin * 2); b_off[k] = take(o.cin * 2); }
  }
  const size_t blob_bytes = align_up(off, 16);
  // Three equal regions per warpgroup, assigned by liveness: the run's input sits in region 0 and every output goes to a
  // free region, region 0 last — so region 0 is idle from the last op that touches the input (or a tensor that had to share
  // its region) onwards and the NEXT patch's input is bulk-copied into it while the remaining ops run.
  region_bytes = align_up(region_bytes, 1024);
  const size_t wg_stride = 3 * region_bytes;
  const int in_t = pr.ops[first].in0;
  auto last_use = [&](int t) {                  // last op of the run that reads tensor t (-1: none); the run's output lives on
    int lu = -1;
    for (int j = first; j <= last; ++j)
      if (pr.ops[j].in0 == t || pr.ops[j].in1 == t) lu = j;
    return lu;
  };
  std::vector<int> region(pr.tensors.size(), -1);
  region[in_t] = 0;
  int last_r0 = -1;
  for (int i = first; i <= last; ++i) {
    const TOp& o = pr.ops[i];
    if (region[o.in0] < 0 || (o.in1 >= 0 && region[o.in1] < 0)) return HN_ERR_UNSUPPORTED;   // reads a tensor from outside the run
    bool busy[3] = {false, false, false};
    busy[region[o.in0]] = true;
    if (o.in1 >= 0) busy[region[o.in1]] = true;
    for (size_t t = 0; t < region.size(); ++t)
      if (region[t] >= 0 && last_use(static_cast<int>(t)) > i) busy[region[t]] = true;
    int r = -1;
    for (int cand : {1, 2, 0})
      if (!busy[cand]) { r = cand; break; }
    if (r < 0) return HN_ERR_UNSUPPORTED;
    for (size_t t = 0; t < region.size(); ++t)
      if (region[t] == r) region[t] = -1;       // a dead tensor's region is reused
    region[o.out] = r;
    // re-derive the inputs' regions for the record below (they cannot have been evicted: they were busy)
    if (region[o.in0] == 0 || (o.in1 >= 0 && region[o.in1] == 0) || r == 0) last_r0 = i - first;
    tl.src_r.push_back(region[o.in0]);
    tl.res_r.push_back(o.in1 >= 0 ? region[o.in1] : -1);
    tl.dst_r.push_back(r);
  }
  // a partial accumulator tile reads up to 2 KB past the end of a source plane: the blob sits behind the last region, so
  // those reads stay inside the CTA's shared memory
  const size_t fixed = align_up(std::max<size_t>(blob_bytes, 2048), 128) + 256 + 1024 /*alignment of the base*/;
  // five or six warpgroups (64 tensor-memory columns and 85 registers each) only for runs without 16 x 16 maps
  int nwg = std::min(h->env.nas_tail_wg, big_map ? 4 : kTailMaxWG);
  while (nwg >= 1 && nwg * wg_stride + fixed > 227 * 1024) --nwg;
  if (nwg < 1) return HN_ERR_UNSUPPORTED;
  tl.first = first; tl.last = last; tl.nwg = nwg;
  tl.last_orig = pr.ops[last].orig;
  TailParams& p = tl.params;
  memset(&p, 0, sizeof(p));
  p.wg_stride = static_cast<int>(wg_stride);
  p.prefetch_after = last_r0 < n - 1 ? last_r0 : -1;
  p.op_base = pr.ops[first].orig >= 0 ? pr.ops[first].orig : first;
  p.launch_id = launch_id & 7;
  p.blob_off = static_cast<int>(nwg * wg_stride);
  p.blob_bytes = static_cast<int>(blob_bytes);
  p.bar_off = static_cast<int>(align_up(p.blob_off + std::max<size_t>(blob_bytes, 2048), 128));
  tl.smem = p.bar_off + 256 + 1024;
  tl.dst_off.assign(n, 0);
  std::vector<uint8_t> blob(std::max<size_t>(blob_bytes, 16), 0);
  p.ones_off = p.blob_off + static_cast<int>(ones_off);
  p.eye_off = p.blob_off + static_cast<int>(eye_off);
  {
    uint16_t* ones = reinterpret_cast<uint16_t*>(blob.data() + ones_off);   // A layout: (k / 8) * 2048 + row * 16 + (k % 8) * 2
    for (int r = 0; r < 128; ++r) ones[r * 8] = ones[r * 8 + 1] = f2h16(1.0f, 0);
    uint16_t* ninf = reinterpret_cast<uint16_t*>(blob.data() + ones_off + 4096);
    for (int j = 0; j < 64; ++j) ninf[j] = 0xFC00;
    uint16_t* eye = reinterpret_cast<uint16_t*>(blob.data() + eye_off);     // B layout: (n / 8) * 256 + (k / 8) * 128 + (n % 8) * 16 + (k % 8) * 2
    for (int d = 0; d < 16; ++d) eye[((d >> 3) * 256 + (d >> 3) * 128 + (d & 7) * 16 + (d & 7) * 2) >> 1] = f2h16(1.0f, 0);
  }
  for (int i = first; i <= last; ++i) {
    const TOp& o = pr.ops[i];
    const int k = i - first;
    TailOp& to = p.ops[k];
    to.kind = o.kind == OP_PW ? TAIL_PW : (o.kind == OP_DW ? TAIL_DW : TAIL_POOL);
    to.shape = tail_op_shape(o);
    to.kernel = o.kernel; to.relu = o.relu;
    to.src_off = static_cast<int>(tl.src_r[k] * region_bytes);
    to.dst_off = static_cast<int>(tl.dst_r[k] * region_bytes);
    to.res_off = tl.res_r[k] >= 0 ? static_cast<int>(tl.res_r[k] * region_bytes) : -1;
    tl.dst_off[k] = to.dst_off;
    to.w_off = p.blob_off + static_cast<int>(w_off[k]);
    to.b_off = p.blob_off + static_cast<int>(b_off[k]);
    tl.out_c.push_back(o.cout); tl.out_h.push_back(o.hout); tl.is_pw.push_back(o.kind == OP_PW);
    uint8_t* b = blob.data();
    if (o.kind == OP_PW) {
      // UMMA no-swizzle K-major image of [W | bias_hi bias_lo 0... | W1] = [cout][K' = cin + 16 + c1w]:
      // element (n, k) at (n / 8) * (K' * 16) + (k / 8) * 128 + (n % 8) * 16 + (k % 8) * 2
      const int c1w = wc1(o);
      const int kp = o.cin + 16 + c1w;
      uint16_t* w = reinterpret_cast<uint16_t*>(b + w_off[k]);
      auto at = [&](int nn, int c) -> uint16_t& { return w[((nn >> 3) * kp * 16 + (c >> 3) * 128 + (nn & 7) * 16 + (c & 7) * 2) >> 1]; };
      for (int nn = 0; nn < o.cout; ++nn) {
        for (int c = 0; c < o.cin; ++c) at(nn, c) = f2h16(o.w[static_cast<size_t>(nn) * o.cin + c], 0);
        const float bias = o.b[nn];
        const __half hi = __float2half_rn(bias);
        at(nn, o.cin) = *reinterpret_cast<const uint16_t*>(&hi);
        at(nn, o.cin + 1) = f2h16(bias - __half2float(hi), 0);
        for (int c = 0; c < c1w; ++c) at(nn, o.cin + 16 + c) = f2h16(o.w1[static_cast<size_t>(nn) * c1w + c], 0);
      }
    } else if (o.kind == OP_DW) {
      uint16_t* w = reinterpret_cast<uint16_t*>(b + w_off[k]);
      for (int j = 0; j < o.kernel * o.kernel * o.cin; ++j) w[j] = f2h16(o.w[j], 0);
      uint16_t* bb = reinterpret_cast<uint16_t*>(b + b_off[k]);
      for (int j = 0; j < o.cin; ++j) bb[j] = f2h16(o.b[j], 0);
    }
  }
  // a pointwise conv whose output is read only by the stride-2 depthwise conv / max-pool right behind it writes the parity layout
  for (int i = first + 1; i <= last; ++i) {
    const TOp& o = pr.ops[i];
    const TOp& pv = pr.ops[i - 1];
    bool only_reader = true;
    for (size_t j = 0; j < pr.ops.size(); ++j)
      if (static_cast<int>(j) != i && (pr.ops[j].in0 == pv.out || pr.ops[j].in1 == pv.out)) only_reader = false;
    if ((o.kind == OP_DW || o.kind == OP_MAXPOOL) && o.stride == 2 && (o.hin == 16 || o.hin == 8) && pv.kind == OP_PW && pv.out == o.in0 &&
        only_reader && pr.head_in != pv.out)
      p.ops[i - first].parity = p.ops[i - 1 - first].parity = 1;
  }
  const TOp& of = pr.ops[first];
  p.in_off = 0;
  p.in_bytes = pr.tensors[in_t].first * pr.tensors[in_t].second * pr.tensors[in_t].second * 2;
  (void)of;
  HN_CUDA(cudaMalloc(&tl.blob, blob.size()));
  HN_CUDA(cudaMemcpy(tl.blob, blob.data(), blob.size(), cudaMemcpyHostToDevice));
  p.blob = reinterpret_cast<const uint4*>(tl.blob);
  return HN_OK;
}

// Cuts `pr` into tail launches (all of it or nothing). A launch boundary needs exactly one tensor crossing it.
static int tail_partition(hn_handle* h, const TProg& pr, std::vector<NasTail>& tails) {
  tails.clear();
  const int n = static_cast<int>(pr.ops.size());
  if (n == 0) return HN_OK;
  for (const TOp& o : pr.ops)
    if (tail_op_shape(o) < 0) return HN_OK;
  auto tensor_bytes = [&](int t) { return static_cast<size_t>(pr.tensors[t].first) * pr.tensors[t].second * pr.tensors[t].second; };
  // only op k's output may be read behind op k (by later ops or by the head)
  auto single_crossing = [&](int k) {
    for (int j = 0; j <= k; ++j) {
      const int t = pr.ops[j].out;
      if (j == k) continue;
      for (int m = k + 1; m < n; ++m)
        if (pr.ops[m].in0 == t || pr.ops[m].in1 == t) return false;
      if (pr.head_in == t) return false;
    }
    const int t0 = pr.ops[0].in0;   // the front stage's output
    for (int m = k + 1; m < n; ++m)
      if (pr.ops[m].in0 == t0 || pr.ops[m].in1 == t0) return false;
    return true;
  };
  std::vector<std::pair<int, int>> runs;
  int start = 0;
  for (int i = 0; i < n; ++i) {
    bool cut = i == n - 1;
    if (!cut && h->env.nas_tail_cut > 0) {
      const size_t in_b = tensor_bytes(pr.ops[start].in0), cut_b = tensor_bytes(pr.ops[i].out);
      cut = cut_b * h->env.nas_tail_cut <= in_b && n - 1 - i >= h->env.nas_tail_minops && single_crossing(i);
    }
    if (cut) { runs.emplace_back(start, i); start = i + 1; }
  }
  for (auto& r : runs) {
    NasTail tl;
    const int rc = tail_build(h, pr, r.first, r.second, static_cast<int>(tails.size()), tl);
    if (rc != HN_OK) {
      for (auto& t2 : tails) cudaFree(t2.blob);
      tails.clear();
      return rc == HN_ERR_UNSUPPORTED ? HN_OK : rc;
    }
    tails.push_back(tl);
  }
  return HN_OK;
}

template <int NWG>
static int launch_tail_cfg(const TailParams& p, size_t smem, int sm_count, cudaStream_t s) {
  auto kern = nas_tail_kernel<NWG>;
  static DeviceOnce attr_once;
  if (attr_once.first_time()) HN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  if (p.n <= 0) return HN_OK;
  kern<<<std::min((p.n + NWG - 1) / NWG, sm_count), NWG * 128, smem, s>>>(p);
  HN_CUDA(cudaGetLastError());
  count_launch();
  return HN_OK;
}

// ops [tl.first, end] of the run for n patches; `out` receives the output of op `end` (channel-planar or NHWC)
static int launch_tail(const NasTail& tl, const uint16_t* in, uint16_t* out, int out_planar, int n, int end, int sm_count, cudaStream_t s) {
  TailParams p = tl.params;
  const int k = end - tl.first;
  p.in = in;
  p.out = out;
  p.n = n;
  p.n_ops = k + 1;
  p.out_off = tl.dst_off[k];
  if (tl.is_pw[k]) p.ops[k].parity = 0;   // a run cut short behind the producer (activation dump) stores plain rows
  p.out_planar = out_planar;
  p.out_pix = tl.out_h[k] * tl.out_h[k];
  p.out_planes_log2 = ilog2(tl.out_c[k] / 8);
  switch (tl.nwg) {
    case 1: return launch_tail_cfg<1>(p, tl.smem, sm_count, s);
    case 2: return launch_tail_cfg<2>(p, tl.smem, sm_count, s);
    case 3: return launch_tail_cfg<3>(p, tl.smem, sm_count, s);
    case 4: return launch_tail_cfg<4>(p, tl.smem, sm_count, s);
    case 5: return launch_tail_cfg<5>(p, tl.smem, sm_count, s);
    default: return launch_tail_cfg<6>(p, tl.smem, sm_count, s);
  }
}

// Runs ops [0, last_op] of the packed program for `n` patches (n <= chunk).
static int run_nas_ops(hn_handle* h, NasState* st, const char* src, int in_dtype, int n, long long off, int last_op, cudaStream_t s) {
  const int bf = st->act_bf16;
  {
      int first = 0;
      if (st->front_img && last_op >= st->front_ops - 1 && h->env.nas_front) {
        const hn_nas_op &o0 = st->ops[0], &ol = st->ops[st->front_ops - 1];
        const int nxt = st->front_ops;
        const hn_nas_op& on = st->ops[nxt];
        if (st->front_fdw && nxt <= last_op) {
          HN_TRY(launch_front_pw_dw(src, in_dtype, st->slot[on.dst], st->params + o0.w_off, st->params + o0.b_off, st->front_img,
                                    st->front_bias2, st->front_fdw, on.kind == OP_DW ? st->params + on.w_off : nullptr,
                                    on.kind == OP_DW ? st->params + on.b_off : nullptr, on.relu, n, h->sm_count, s,
                                    /*out_planar=*/nxt < last_op && st->tail_of_op[nxt + 1] >= 0));
          first = nxt + 1;
        } else {
          HN_TRY(launch_front_pw(src, in_dtype, st->slot[ol.dst], st->front_tm, st->params + o0.w_off, st->params + o0.b_off, st->front_img,
                                 st->front_bias2, n, bf, h->sm_count, s));
          first = st->front_ops;
        }
      }
      const int n_total = static_cast<int>(st->ops.size());
      for (int i = first; i <= last_op; ++i) {
        const hn_nas_op& o = st->ops[i];
        if (i == st->tail_first && last_op == n_total - 1 && !st->ftails.empty()) {
          // the forward: folded form, launches chained through the slots, the last one writes the head GEMM's rows
          const uint16_t* cur = st->slot[st->ops[i].src];
          int cur_slot = st->ops[i].src;
          for (size_t k = 0; k < st->ftails.size(); ++k) {
            const NasTail& tl = st->ftails[k];
            const bool lastl = k + 1 == st->ftails.size();
            const int nxt_slot = (cur_slot + 1) % 3;
            uint16_t* dst = lastl ? st->head_in + static_cast<size_t>(off) * st->headf_k : st->slot[nxt_slot];
            HN_TRY(launch_tail(tl, cur, dst, 1, n, tl.last, h->sm_count, s));
            cur = dst;
            cur_slot = nxt_slot;
          }
          break;
        }
        if (st->tail_of_op[i] >= 0) {
          // plain form: packed ops [i, end]; a run that ends right before the head writes the head GEMM's rows
          const NasTail& tl = st->tails[st->tail_of_op[i]];
          const int end = std::min(tl.last + st->tail_first, last_op);
          const bool to_head = end == n_total - 2 && last_op == n_total - 1;
          uint16_t* dst = to_head ? st->head_in + static_cast<size_t>(off) * st->head_k : st->slot[st->ops[end].dst];
          // channel-planar interchange towards the next tail launch / the head GEMM (permuted weight K order); a run that
          // stops here (activation dump) writes NHWC like every per-op kernel
          const int planar = (to_head && st->head_planar) || (end == tl.last + st->tail_first && last_op > end && st->tail_of_op[end + 1] >= 0);
          HN_TRY(launch_tail(tl, st->slot[st->ops[tl.first + st->tail_first].src], dst, planar, n, end - st->tail_first, h->sm_count, s));
          i = to_head ? end + 1 : end;
          continue;
        }
        switch (o.kind) {
          case OP_STEM: {
            HN_TRY(launch_l1(src, in_dtype, st->slot[o.dst], st->params + o.w_off, st->params + o.b_off, nullptr, n, bf, h->sm_count, s));
            break;
          }
          case OP_PW: {
            PwParams p = st->pw[i];
            p.total_rows = static_cast<long long>(n) * o.hin * o.hin / p.row_div;
            p.num_tiles = static_cast<int>((p.total_rows + kTileM - 1) / kTileM) * p.n_tiles;
            HN_TRY(launch_pw(p, p.nt, p.kcb, h->sm_count, s));
            break;
          }
          case OP_DW: {
            const bool strip = (o.kernel == 3 || o.kernel == 5) && (o.stride == 1 || o.stride == 2) && o.hout % 4 == 0;
            const long long total = static_cast<long long>(n) * o.hout * (strip ? o.hout / 4 : o.hout) * (o.cin / 8);
            const int grid = static_cast<int>(std::min<long long>((total + 255) / 256, h->sm_count * 16LL));
            const uint16_t* src = st->slot[o.src];
            uint16_t* dst = st->slot[o.dst];
            const float* wv = st->params + o.w_off;
            const float* bv = st->params + o.b_off;
            // shared-memory kernel whenever one unit of two whole maps fits next to the weights (227 KB): every depthwise
            // shape of SEARCH_SPACE2 except the 32 x 32 input maps of a layer-0 block wider than 32 channels (e3 / s4 / e6:
            // 96-192 channels, 388-788 KB), which fall through to the register-strip kernel below
            if (strip && h->env.nas_dw_smem) {
              const size_t map_bytes = static_cast<size_t>(o.hin) * o.hin * o.cin * 2;
              // 5x5 stride 1 is bound by the fp32 pipe + unpack instructions: strips of 8 rows re-use each loaded and
              // unpacked input vector for more taps (12 rows for 8 outputs instead of 8 for 4)
              const int sh = (o.kernel == 5 && o.stride == 1 && o.hout % 8 == 0 && h->env.nas_dw_sh8) ? 8 : 4;
              const int items = (o.hout / sh) * o.hout * (o.cin / 8);
              int G = std::max(1, 256 / items);
              const size_t w_bytes = ((static_cast<size_t>(o.kernel) * o.kernel + 1) * o.cin * 4 + 127) & ~size_t(127);
              while (G > 1 && w_bytes + 2 * G * map_bytes + 32 > 110 * 1024) G >>= 1;
              const size_t smem = w_bytes + 2 * G * map_bytes + 32;
              if (smem <= 227 * 1024) {
                const int units = (n + G - 1) / G;
                // resident CTAs per SM: shared memory, and registers for the 8-row variant (~176 per thread)
                const bool f32_math = bf || h->env.nas_dw_f32;   // the 8-row fp32 variant needs ~176 registers per thread, the half2 one ~110
                const int per_sm = (sh == 8 && f32_math) ? 1 : std::max(1, std::min(sh == 8 ? 2 : 4, static_cast<int>((227 * 1024) / (smem + 1024))));
                const int sgrid = std::min(units, h->sm_count * per_sm);
#define HN_DW_SMEM(KK, SS, SHH, BF)                                                                                   \
  do {                                                                                                                \
    static DeviceOnce once;                                                                                           \
    if (once.first_time())                                                                                            \
      HN_CUDA(cudaFuncSetAttribute(dw_conv_smem_kernel<KK, SS, SHH, BF>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)); \
    dw_conv_smem_kernel<KK, SS, SHH, BF><<<sgrid, 256, smem, s>>>(src, dst, wv, bv, n, o.cin, o.hin, o.hout, G, o.relu); \
  } while (0)
#define HN_DW_SMEM_H2(KK, SS, SHH)                                                                                    \
  do {                                                                                                                \
    static DeviceOnce once;                                                                                           \
    if (once.first_time())                                                                                            \
      HN_CUDA(cudaFuncSetAttribute(dw_conv_smem_h2_kernel<KK, SS, SHH>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)); \
    dw_conv_smem_h2_kernel<KK, SS, SHH><<<sgrid, 256, smem, s>>>(src, dst, wv, bv, n, o.cin, o.hin, o.hout, G, o.relu); \
  } while (0)
#define HN_DW_SMEM_T(KK, SS, SHH) do { if (bf) HN_DW_SMEM(KK, SS, SHH, true); else if (h->env.nas_dw_f32) HN_DW_SMEM(KK, SS, SHH, false); else HN_DW_SMEM_H2(KK, SS, SHH); } while (0)
                if (o.kernel == 3 && o.stride == 1) HN_DW_SMEM_T(3, 1, 4);
                else if (o.kernel == 3) HN_DW_SMEM_T(3, 2, 4);
                else if (o.stride == 1 && sh == 8) HN_DW_SMEM_T(5, 1, 8);
                else if (o.stride == 1) HN_DW_SMEM_T(5, 1, 4);
                else HN_DW_SMEM_T(5, 2, 4);
#undef HN_DW_SMEM_T
#undef HN_DW_SMEM_H2
#undef HN_DW_SMEM
                HN_CUDA(cudaGetLastError());
                count_launch();
                break;
              }
            }
#define HN_DW_STRIP(KK, SS) dw_conv_strip_kernel<KK, SS><<<grid, 256, 0, s>>>(src, dst, wv, bv, n, o.cin, o.hin, o.hout, o.relu, bf)
            if (!strip) dw_conv_kernel<<<grid, 256, 0, s>>>(src, dst, wv, bv, n, o.cin, o.hin, o.hout, o.kernel, o.stride, o.relu, bf);
            else if (o.kernel == 3 && o.stride == 1) HN_DW_STRIP(3, 1);
            else if (o.kernel == 3) HN_DW_STRIP(3, 2);
            else if (o.stride == 1) HN_DW_STRIP(5, 1);
            else HN_DW_STRIP(5, 2);
#undef HN_DW_STRIP
            HN_CUDA(cudaGetLastError());
            count_launch();
            break;
          }
          case OP_MAXPOOL: {
            const long long total = static_cast<long long>(n) * o.hout * o.hout * (o.cin / 8);
            const int grid = static_cast<int>(std::min<long long>((total + 255) / 256, h->sm_count * 16LL));
            {
              const size_t map_bytes = static_cast<size_t>(o.hin) * o.hin * o.cin * 2;
              const int items = (o.hout / 4) * o.hout * (o.cin / 8);
              int G = items > 0 ? std::max(1, 256 / items) : 1;
              while (G > 1 && 2 * G * map_bytes + 48 > 110 * 1024) G >>= 1;
              const size_t smem = 2 * G * map_bytes + 48;
              if (o.hout % 4 == 0 && smem <= 227 * 1024 && h->env.nas_dw_smem) {
                const int units = (n + G - 1) / G;
                const int per_sm = std::max(1, std::min(4, static_cast<int>((227 * 1024) / (smem + 1024))));
                const int sgrid = std::min(units, h->sm_count * per_sm);
                static DeviceOnce once;
                if (once.first_time()) {
                  HN_CUDA(cudaFuncSetAttribute(maxpool_smem_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
                  HN_CUDA(cudaFuncSetAttribute(maxpool_smem_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
                }
                if (bf) maxpool_smem_kernel<true><<<sgrid, 256, smem, s>>>(st->slot[o.src], st->slot[o.dst], n, o.cin, o.hin, o.hout, G);
                else maxpool_smem_kernel<false><<<sgrid, 256, smem, s>>>(st->slot[o.src], st->slot[o.dst], n, o.cin, o.hin, o.hout, G);
                HN_CUDA(cudaGetLastError());
                count_launch();
                break;
              }
            }
            maxpool_kernel<<<grid, 256, 0, s>>>(st->slot[o.src], st->slot[o.dst], n, o.cin, o.hin, o.hout, bf);
            HN_CUDA(cudaGetLastError());
            count_launch();
            break;
          }
          case OP_SE: {
            se_kernel<<<std::min(n, h->sm_count * 8), 256, 0, s>>>(st->slot[o.src], n, o.cin, o.hin, o.mid, st->params + o.w_off,
                                                                  st->params + o.b_off, st->params + o.w2_off,
                                                                  st->params + o.b2_off, bf);
            HN_CUDA(cudaGetLastError());
            count_launch();
            break;
          }
          case OP_HEAD: {
            HN_CUDA(cudaMemcpyAsync(st->head_in + static_cast<size_t>(off) * st->head_k, st->slot[o.src],
                                    static_cast<size_t>(n) * st->head_k * 2, cudaMemcpyDeviceToDevice, s));
            break;
          }
        }
      }
    }
  return HN_OK;
}
}  // namespace hn

using namespace hn;

extern "C" int hn_pack_nas(hn_handle* h, const hn_nas_op* ops, int n_ops, const float* params, long long n_params,
                           int act_dtype) {
  HN_REQUIRE(h && ops && params && n_ops >= 2 && n_params > 0, "hn_pack_nas: bad argument");
  HN_REQUIRE(act_dtype == HN_F16 || act_dtype == HN_BF16, "hn_pack_nas: act_dtype must be HN_F16 or HN_BF16");
  HN_REQUIRE(ops[0].kind == OP_STEM && ops[0].cout == 32 && ops[0].hin == 32, "hn_pack_nas: first op must be the 1->32 stem");
  HN_REQUIRE(ops[n_ops - 1].kind == OP_HEAD && ops[n_ops - 1].cout == 128, "hn_pack_nas: last op must be the 128-d head");
  const int bf = act_dtype == HN_BF16;
  // same ordering rule as hn_pack_hardnet: drain every stream before the old net is freed, and again once the copies landed
  HN_CUDA(cudaDeviceSynchronize());
  nas_state_free(h->nas);
  h->nas = nullptr;
  NasState* st = new NasState();
  auto fail = [&](int code) { nas_state_free(st); return code; };
  st->act_bf16 = bf;
  st->ops.assign(ops, ops + n_ops);
  st->pw.resize(n_ops);
  st->w16_off.assign(n_ops, 0);
  // validate + size
  size_t w16_total = 0;
  for (int i = 0; i < n_ops; ++i) {
    const hn_nas_op& o = ops[i];
    auto in_blob = [&](long long off, long long n) { return off >= 0 && off + n <= n_params; };
    if (o.kind != OP_STEM && (o.src < 0 || o.src > 2)) { set_error("hn_pack_nas: op %d has a bad src slot", i); return fail(HN_ERR_INVALID); }
    if (o.kind != OP_HEAD && (o.dst < 0 || o.dst > 2)) { set_error("hn_pack_nas: op %d has a bad dst slot", i); return fail(HN_ERR_INVALID); }
    if (o.kind != OP_STEM) st->slot_elems = std::max(st->slot_elems, static_cast<size_t>(o.cin) * o.hin * o.hin);
    if (o.kind != OP_HEAD) st->slot_elems = std::max(st->slot_elems, static_cast<size_t>(o.cout) * o.hout * o.hout);
    bool ok = true;
    switch (o.kind) {
      case OP_STEM: ok = in_blob(o.w_off, 9 * 32) && in_blob(o.b_off, 32); break;
      case OP_PW:
        ok = o.cin % 32 == 0 && o.cout % 32 == 0 && o.cin <= 512 && o.cout <= 512 && in_blob(o.w_off, 1LL * o.cin * o.cout) &&
             in_blob(o.b_off, o.cout) && o.res >= -1 && o.res <= 2 && o.res != o.dst && o.src != o.dst;
        ok = ok && (o.hin * o.hin) % 2 == 0;
        st->w16_off[i] = w16_total;
        w16_total += static_cast<size_t>(o.cin) * o.cout * (pw_row_paired(o) ? 4 : 1);
        break;
      case OP_DW:
        ok = o.cin == o.cout && o.cin % 8 == 0 && (o.kernel == 3 || o.kernel == 5) && (o.stride == 1 || o.stride == 2) &&
             o.hout * o.stride == o.hin && in_blob(o.w_off, 1LL * o.kernel * o.kernel * o.cin) && in_blob(o.b_off, o.cin) &&
             o.src != o.dst;
        break;
      case OP_MAXPOOL: ok = o.cin == o.cout && o.cin % 8 == 0 && o.hout * 2 == o.hin && o.src != o.dst; break;
      case OP_SE:
        ok = o.cin <= 512 && o.mid <= 128 && o.cin % 2 == 0 && o.src == o.dst && in_blob(o.w_off, 1LL * o.mid * o.cin) &&
             in_blob(o.b_off, o.mid) && in_blob(o.w2_off, 1LL * o.mid * o.cin) && in_blob(o.b2_off, o.cin);
        break;
      case OP_HEAD: {
        const long long K = 1LL * o.kernel * o.kernel * o.cin;
        ok = o.kernel == o.hin && K % 128 == 0 && in_blob(o.w_off, 128 * K) && in_blob(o.b_off, 128);
        st->w16_off[i] = w16_total;
        w16_total += static_cast<size_t>(128) * K;
        st->head_k = static_cast<int>(K);
        break;
      }
      default: ok = false;
    }
    if (!ok) { set_error("hn_pack_nas: op %d (kind %d) failed validation", i, o.kind); return fail(HN_ERR_INVALID); }
  }
#define HN_CUDA_N(expr)                                                                          \
  do {                                                                                           \
    cudaError_t e__ = (expr);                                                                    \
    if (e__ != cudaSuccess) {                                                                    \
      set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__));           \
      return fail(HN_ERR_CUDA);                                                                  \
    }                                                                                            \
  } while (0)
  HN_CUDA_N(cudaMalloc(&st->params, static_cast<size_t>(n_params) * sizeof(float)));
  HN_CUDA_N(cudaMemcpy(st->params, params, static_cast<size_t>(n_params) * sizeof(float), cudaMemcpyHostToDevice));
  {
    std::vector<uint16_t> w16(w16_total);
    for (int i = 0; i < n_ops; ++i) {
      const hn_nas_op& o = ops[i];
      if (o.kind == OP_PW && pw_row_paired(o)) {   // [[W, 0], [0, W]] as [2 C_out][64]; the vector is zero-initialised
        for (int hh = 0; hh < 2; ++hh)
          for (int co = 0; co < o.cout; ++co)
            for (int ci = 0; ci < 32; ++ci)
              w16[st->w16_off[i] + static_cast<size_t>(hh * o.cout + co) * 64 + hh * 32 + ci] = f2h16(params[o.w_off + co * 32 + ci], bf);
        continue;
      }
      const size_t n = o.kind == OP_PW ? static_cast<size_t>(o.cin) * o.cout : o.kind == OP_HEAD ? static_cast<size_t>(128) * st->head_k : 0;
      for (size_t j = 0; j < n; ++j) w16[st->w16_off[i] + j] = f2h16(params[o.w_off + j], bf);
    }
    HN_CUDA_N(cudaMalloc(&st->w16, std::max<size_t>(w16_total, 1) * 2));
    HN_CUDA_N(cudaMemcpy(st->w16, w16.data(), w16_total * 2, cudaMemcpyHostToDevice));
  }
  {
    const size_t cap = (size_t(4) << 30) / (6 * st->slot_elems);
    st->chunk = static_cast<int>(std::min<size_t>(h->chunk, std::max<size_t>(cap, 64))) & ~1;
  }
  const size_t slot_bytes = static_cast<size_t>(st->chunk) * st->slot_elems * 2;
  for (int k = 0; k < 3; ++k) {
    HN_CUDA_N(cudaMalloc(&st->slot[k], slot_bytes));
    HN_CUDA_N(cudaMemset(st->slot[k], 0, slot_bytes));
  }
  // stem -> pointwise 32 -> 32 + ReLU (the expansion conv of an expansion-1 block): one fused front-kernel launch
  if (ops[1].kind == OP_PW && ops[1].cin == 32 && ops[1].cout == 32 && ops[1].hin == 32 && ops[1].relu && ops[1].res < 0 &&
      ops[1].src == ops[0].dst) {
    bool stem_reused = false;                  // nothing later may read the stem output, which no longer exists
    for (int i = 2; i < n_ops && !stem_reused; ++i) {
      if (ops[i].kind != OP_HEAD && ops[i].dst == ops[0].dst) break;   // slot overwritten: later readers see the new tensor
      stem_reused = ops[i].src == ops[0].dst || (ops[i].kind == OP_PW && ops[i].res == ops[0].dst);
    }
    if (!stem_reused) {
      std::vector<uint16_t> w16(32 * 32), img;
      for (int j = 0; j < 32 * 32; ++j) w16[j] = f2h16(params[ops[1].w_off + j], bf);
      front_pw_weight_image(w16.data(), img);
      memcpy(st->front_bias2, params + ops[1].b_off, sizeof(st->front_bias2));
      HN_CUDA_N(cudaMalloc(&st->front_img, img.size() * 2));
      HN_CUDA_N(cudaMemcpy(st->front_img, img.data(), img.size() * 2, cudaMemcpyHostToDevice));
      st->front_ops = 2;
    }
  }
  if (!st->front_img) {
    // The stem ALONE also runs on the fused front kernel, with an identity second stage (W = I, bias 0; the stem output is
    // >= 0, so the second ReLU and the 16-bit re-rounding change nothing): its whole-patch stage-1 issue and TMA output
    // stores make it 1.5x faster than the stand-alone stem kernel (0.27 vs 0.42 ms per 18 944 patches).
    std::vector<uint16_t> w16(32 * 32, 0), img;
    for (int c = 0; c < 32; ++c) w16[c * 32 + c] = f2h16(1.0f, bf);
    front_pw_weight_image(w16.data(), img);
    memset(st->front_bias2, 0, sizeof(st->front_bias2));
    HN_CUDA_N(cudaMalloc(&st->front_img, img.size() * 2));
    HN_CUDA_N(cudaMemcpy(st->front_img, img.data(), img.size() * 2, cudaMemcpyHostToDevice));
    st->front_ops = 1;
  }
  // the op behind the front stage, if it is the block's stride-2 depthwise conv (or the Identity's max-pool) on the
  // 32 x 32 x 32 tensor, runs inside the front kernel too (fp16 activations): 64 KB/patch never reach HBM
  if (!bf && h->env.nas_front_dw && h->env.nas_front && st->front_ops < n_ops - 1) {
    const hn_nas_op& o = ops[st->front_ops];
    const hn_nas_op& prev = ops[st->front_ops - 1];
    const bool shape_ok = o.cin == 32 && o.cout == 32 && o.hin == 32 && o.hout == 16 && o.stride == 2 && o.src == prev.dst;
    const int fdw = (o.kind == OP_DW && (o.kernel == 3 || o.kernel == 5)) ? o.kernel : (o.kind == OP_MAXPOOL ? 1 : 0);
    bool reused = false;               // nothing later may read the pointwise output, which no longer exists
    for (int i = st->front_ops + 1; i < n_ops && !reused; ++i) {
      if (ops[i].kind != OP_HEAD && ops[i].dst == prev.dst) break;
      reused = ops[i].src == prev.dst || (ops[i].kind == OP_PW && ops[i].res == prev.dst);
    }
    if (shape_ok && fdw && !reused) st->front_fdw = fdw;
  }
  HN_CUDA_N(cudaMalloc(&st->head_in, static_cast<size_t>(h->head_rows) * st->head_k * 2));
  HN_CUDA_N(cudaMemset(st->head_in, 0, static_cast<size_t>(h->head_rows) * st->head_k * 2));
#undef HN_CUDA_N
  // static descriptors
  for (int i = 0; i < n_ops; ++i) {
    const hn_nas_op& o = ops[i];
    if (o.kind == OP_PW) {
      PwParams& p = st->pw[i];
      memset(&p, 0, sizeof(p));
      const int row_div = pw_row_paired(o) ? 2 : 1;
      const int cin = o.cin * row_div, cout = o.cout * row_div;
      const int kcb = (cin % 64 == 0) ? 128 : 64;
      const int kc = kcb / 2;
      const int nt = pick_nt(cout);
      const uint64_t rows_cap = static_cast<uint64_t>(st->chunk) * o.hin * o.hin / row_div;
      const uint64_t dimsA[2] = {static_cast<uint64_t>(cin), rows_cap};
      const uint64_t strA[1] = {static_cast<uint64_t>(cin) * 2};
      const uint32_t boxA[2] = {static_cast<uint32_t>(kc), static_cast<uint32_t>(kTileM)};
      int rc = make_tmap_16bit(&p.tmA, st->slot[o.src], 2, dimsA, strA, boxA, kcb);
      if (rc != HN_OK) return fail(rc);
      const uint64_t dimsB[2] = {static_cast<uint64_t>(cin), static_cast<uint64_t>(cout)};
      const uint32_t boxB[2] = {static_cast<uint32_t>(kc), static_cast<uint32_t>(nt)};
      rc = make_tmap_16bit(&p.tmB, st->w16 + st->w16_off[i], 2, dimsB, strA, boxB, kcb);
      if (rc != HN_OK) return fail(rc);
      if (nt == 32 || nt == 64 || nt == 128) {
        const int boxc = std::min(nt, 64);
        const uint64_t dimsO[2] = {static_cast<uint64_t>(cout), rows_cap};
        const uint64_t strO[1] = {static_cast<uint64_t>(cout) * 2};
        const uint32_t boxO[2] = {static_cast<uint32_t>(boxc), 32};
        rc = make_tmap_16bit(&p.tmO, st->slot[o.dst], 2, dimsO, strO, boxO, boxc * 2);
        if (rc != HN_OK) return fail(rc);
        if (o.res >= 0) {
          rc = make_tmap_16bit(&p.tmR, st->slot[o.res], 2, dimsO, strO, boxO, boxc * 2);
          if (rc != HN_OK) return fail(rc);
        }
      }
      p.bias = st->params + o.b_off;
      p.res = o.res >= 0 ? st->slot[o.res] : nullptr;
      p.out = st->slot[o.dst];
      p.n_tiles = cout / nt;
      p.num_kb = cin / kc;
      p.cout = cout;
      p.bias_n = o.cout;
      p.nt = nt;
      p.kcb = kcb;
      p.row_div = row_div;
      p.relu = o.relu;
      p.act_bf16 = bf;
    } else if (o.kind == OP_HEAD) {
      TcParams& p = st->head;
      memset(&p, 0, sizeof(p));
      const uint64_t K = static_cast<uint64_t>(st->head_k);
      const uint64_t dimsA[2] = {K, static_cast<uint64_t>(h->head_rows)};
      const uint64_t strA[1] = {K * 2};
      const uint32_t boxA[2] = {64, static_cast<uint32_t>(kTileM)};
      int rc = make_tmap_16bit(&p.tmA[0], st->head_in, 2, dimsA, strA, boxA, 128);
      if (rc != HN_OK) return fail(rc);
      const uint64_t dimsB[2] = {K, 128};
      const uint32_t boxB[2] = {64, 128};
      rc = make_tmap_16bit(&p.tmB, st->w16 + st->w16_off[i], 2, dimsB, strA, boxB, 128);
      if (rc != HN_OK) return fail(rc);
      p.num_k_stages = static_cast<int>(K / (64 * kHeadG));
      p.bias = st->params + o.b_off;
      p.l2_eps = 0.f;  // torch.norm without eps (model_supernet.py:84)
      p.act_bf16 = bf;
    }
  }
  if (st->front_img) {
    const uint64_t dimsO[2] = {32, static_cast<uint64_t>(st->chunk) * 1024};
    const uint64_t strO[1] = {64};
    const uint32_t boxO[2] = {32, 32};
    const int rc = make_tmap_16bit(&st->front_tm, st->slot[ops[st->front_ops - 1].dst], 2, dimsO, strO, boxO, 64);
    if (rc != HN_OK) return fail(rc);
  }
  {
    int rc = HN_OK;
    // warpgroup-per-patch tail launches behind the fused front stage (fp16 activations, every op of a supported shape)
    st->tail_of_op.assign(n_ops, -1);
    st->tail_first = st->front_ops + 1;
    if (h->env.nas_tail && !bf && st->front_fdw && h->env.nas_front && st->tail_first <= n_ops - 2) {
      TProg plain;
      if (tail_prog_plain(st->ops, params, st->tail_first, plain)) {
        rc = tail_partition(h, plain, st->tails);
        if (rc != HN_OK) return fail(rc);
      }
      for (size_t k = 0; k < st->tails.size(); ++k)
        for (int i = st->tails[k].first; i <= st->tails[k].last; ++i) st->tail_of_op[st->tail_first + i] = static_cast<int>(k);
      TProg fold;
      if (!st->tails.empty() && h->env.nas_fold && tail_prog_folded(st->ops, params, st->tail_first, fold)) {
        rc = tail_partition(h, fold, st->ftails);
        if (rc != HN_OK) return fail(rc);
      }
      auto planar_head = [&](const TProg& pr, std::vector<uint16_t>& wh) {
        // a tail launch bulk-stores its channel-planar output as the head GEMM's input row: K index
        // plane * (pix * 8) + pixel * 8 + c % 8 instead of NHWC's pixel * C + c
        const int pix = pr.head_pix, C = pr.head_c;
        const size_t K = static_cast<size_t>(pix) * C;
        wh.assign(128 * K, 0);
        for (int nn = 0; nn < 128; ++nn)
          for (int px = 0; px < pix; ++px)
            for (int c = 0; c < C; ++c)
              wh[nn * K + (c >> 3) * (pix * 8) + px * 8 + (c & 7)] = f2h16(pr.head_w[nn * K + static_cast<size_t>(px) * C + c], 0);
      };
      if (!st->tails.empty()) {
        std::vector<uint16_t> wh;
        planar_head(plain, wh);
        if (cudaMemcpy(st->w16 + st->w16_off[n_ops - 1], wh.data(), wh.size() * 2, cudaMemcpyHostToDevice) != cudaSuccess) {
          set_error("hn_pack_nas: head weight upload failed");
          return fail(HN_ERR_CUDA);
        }
        st->head_planar = 1;
      }
      if (!st->ftails.empty()) {
        std::vector<uint16_t> wh;
        planar_head(fold, wh);
        st->headf_k = fold.head_pix * fold.head_c;
        if (cudaMalloc(&st->headf_w, wh.size() * 2) != cudaSuccess || cudaMalloc(&st->headf_b, 128 * sizeof(float)) != cudaSuccess ||
            cudaMemcpy(st->headf_w, wh.data(), wh.size() * 2, cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaMemcpy(st->headf_b, fold.head_b.data(), 128 * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess) {
          set_error("hn_pack_nas: folded head upload failed");
          return fail(HN_ERR_CUDA);
        }
        TcParams& hp = st->headf;
        hp = st->head;
        const uint64_t K = static_cast<uint64_t>(st->headf_k);
        const uint64_t dimsA[2] = {K, static_cast<uint64_t>(h->head_rows)};
        const uint64_t strA[1] = {K * 2};
        const uint32_t boxA[2] = {64, static_cast<uint32_t>(kTileM)};
        rc = make_tmap_16bit(&hp.tmA[0], st->head_in, 2, dimsA, strA, boxA, 128);
        if (rc != HN_OK) return fail(rc);
        const uint64_t dimsB[2] = {K, 128};
        const uint32_t boxB[2] = {64, 128};
        rc = make_tmap_16bit(&hp.tmB, st->headf_w, 2, dimsB, strA, boxB, 128);
        if (rc != HN_OK) return fail(rc);
        hp.num_k_stages = static_cast<int>(K / (64 * kHeadG));
        hp.bias = st->headf_b;
      }
    }
  }
  if (cudaDeviceSynchronize() != cudaSuccess) {
    set_error("hn_pack_nas: cudaDeviceSynchronize failed");
    return fail(HN_ERR_CUDA);
  }
  h->nas = st;
  return HN_OK;
}

extern "C" int hn_forward_nas(hn_handle* h, const void* patches, int in_dtype, long long B, void* desc_out, int out_dtype,
                              void* stream) {
  HN_REQUIRE(h, "hn_forward_nas: NULL handle");
  if (!h->nas) {
    set_error("hn_forward_nas: no NAS net packed (call hn_pack_nas first)");
    return HN_ERR_STATE;
  }
  HN_REQUIRE(B >= 0, "hn_forward_nas: negative batch");
  HN_REQUIRE(in_dtype == HN_F32 || in_dtype == HN_U8, "hn_forward_nas: in_dtype must be HN_F32 or HN_U8");
  HN_REQUIRE(out_dtype == HN_F32 || out_dtype == HN_F16 || out_dtype == HN_BF16 || out_dtype == HN_F8E4M3, "hn_forward_nas: bad out_dtype");
  if (B == 0) return HN_OK;
  HN_REQUIRE(patches && desc_out, "hn_forward_nas: NULL data pointer");
  NasState* st = h->nas;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t in_elem = in_dtype == HN_F32 ? 4 : 1;
  const size_t out_elem = out_dtype == HN_F32 ? 4 : out_dtype == HN_F8E4M3 ? 1 : 2;
  const int n_ops = static_cast<int>(st->ops.size());
  for (long long base = 0; base < B; base += h->head_rows) {
    const long long nb = std::min<long long>(h->head_rows, B - base);
    for (long long off = 0; off < nb; off += st->chunk) {
      const int n = static_cast<int>(std::min<long long>(st->chunk, nb - off));
      const char* src = static_cast<const char*>(patches) + static_cast<size_t>(base + off) * 1024 * in_elem;
      HN_TRY(run_nas_ops(h, st, src, in_dtype, n, off, n_ops - 1, s));
    }
    TcParams p = st->ftails.empty() ? st->head : st->headf;
    p.total_rows = nb;
    p.num_tiles = static_cast<int>((nb + kTileM - 1) / kTileM);
    p.out_dtype = out_dtype;
    p.out = static_cast<char*>(desc_out) + static_cast<size_t>(base) * 128 * out_elem;
    p.partial = h->head_partial;
    HN_TRY(launch_head(p, h->sm_count, s));
  }
  return HN_OK;
}

#ifdef HN_TAIL_TRACE
extern "C" int hn_debug_tail_trace(unsigned long long* out128, int reset) {
  HN_CUDA(cudaDeviceSynchronize());
  HN_CUDA(cudaMemcpyFromSymbol(out128, hn::hn_tail_trace, 128 * sizeof(unsigned long long)));
  if (reset) {
    unsigned long long z[128] = {0};
    HN_CUDA(cudaMemcpyToSymbol(hn::hn_tail_trace, z, sizeof(z)));
  }
  return HN_OK;
}
#endif

extern "C" int hn_nas_plan(hn_handle* h, int* out, int cap) {
  HN_REQUIRE(h, "hn_nas_plan: NULL handle");
  if (!h->nas) {
    set_error("hn_nas_plan: no NAS net packed");
    return HN_ERR_STATE;
  }
  int n = 0;
  // warpgroup-per-patch tail launches of the forward: (first packed op, last packed op, patches in flight per CTA, 0); in the
  // folded form a launch starts / ends at the packed op whose output its first / last op produces
  const bool folded = !h->nas->ftails.empty();
  for (const NasTail& tl : (folded ? h->nas->ftails : h->nas->tails)) {
    if (n < cap && out) {
      out[4 * n] = folded ? tl.params.op_base : tl.first + h->nas->tail_first;
      out[4 * n + 1] = folded ? tl.last_orig : tl.last + h->nas->tail_first;
      out[4 * n + 2] = tl.nwg; out[4 * n + 3] = 0;
    }
    ++n;
  }
  return n;
}

extern "C" int hn_forward_nas_dump(hn_handle* h, const void* patches, int in_dtype, long long B, int op_index, void* act_out,
                                   void* stream) {
  HN_REQUIRE(h && patches && act_out, "hn_forward_nas_dump: NULL argument");
  if (!h->nas) {
    set_error("hn_forward_nas_dump: no NAS net packed");
    return HN_ERR_STATE;
  }
  NasState* st = h->nas;
  HN_REQUIRE(op_index >= 0 && op_index < static_cast<int>(st->ops.size()) - 1, "hn_forward_nas_dump: op_index out of range");
  HN_REQUIRE(B >= 1 && B <= st->chunk, "hn_forward_nas_dump: B must be in [1, chunk=%d]", st->chunk);
  HN_REQUIRE(in_dtype == HN_F32 || in_dtype == HN_U8, "hn_forward_nas_dump: bad in_dtype");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  HN_TRY(run_nas_ops(h, st, static_cast<const char*>(patches), in_dtype, static_cast<int>(B), 0, op_index, s));
  const hn_nas_op& o = st->ops[op_index];
  HN_CUDA(cudaMemcpyAsync(act_out, st->slot[o.dst], static_cast<size_t>(B) * o.cout * o.hout * o.hout * 2,
                          cudaMemcpyDeviceToDevice, s));
  return HN_OK;
}
