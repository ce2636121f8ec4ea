// NAS descriptor net behind the fused front kernel as ONE launch per run of blocks ("tail"): every op between the
// front stage (stem + first pointwise conv + stride-2 depthwise conv / max-pool, front_fused.cuh) and the head GEMM —
// hardnetNAS/fbnet_building_blocks/fbnet_builder.py:455-570 (IRFBlock: pw -> dw -> pwl [+ x]) and :202-228 (Identity:
// max-pool / 1x1 conv), stacked as in hardnetNAS/supernet_functions/model_supernet.py:70-85 — runs with the patch's
// activations resident in shared memory.
//
// The unit of execution is a WARPGROUP, not the CTA (a CTA that steps through the ops of a group of patches pays a CTA-wide
// issue -> commit -> wait -> tcgen05.ld -> store -> barrier latency at every step; DESIGN.md section 4):
// four warps own ONE patch from its load to its store, synchronise only among themselves (named barrier, own mbarrier,
// own 128 tensor-memory columns) and the 3-4 warpgroups of a CTA run independently, so one warpgroup's latency-bound
// tensor-core phase overlaps the others' CUDA-core depthwise phases without any hand-written pipeline. All shapes are
// compile-time (the search space SEARCH_SPACE2 has five stage shapes behind the front kernel, lookup_table_builder.py:18-45),
// so the per-thread work split needs no integer division and every thread of a warpgroup has exactly one depthwise item.
//   PW    1x1 conv: tcgen05 GEMM on the activation IN PLACE (channel-planar [c / 8][pixel][c % 8] = UMMA no-swizzle
//         K-major, SBO 128 B, LBO = plane pitch) against the resident weight image. Bias and residual are added BY THE
//         TENSOR CORE (one K step of a constant "ones" tile against the bias stored as fp16 hi + lo behind the weights;
//         16-channel slices of the block input against a 16 x 16 identity), so the epilogue is only TMEM -> [ReLU] -> fp16
//         -> planar destination. Maps with fewer than 128 pixels issue a full M = 128 tile and ignore the
//         surplus accumulator rows.
//   DW    depthwise k x k (3 | 5, stride 1 | 2) in packed half2 arithmetic, the summation order of dw_conv_smem_h2_kernel
//         (nas.cu); a thread = 8 channels x one output column x a strip of SH rows, SH = C * hout^2 / 1024.
//   POOL  MaxPool2d(3, 2, 1) with packed fp16 maxima.
// fp16 activations, expansion-1 blocks without SE (every recorded architecture: wang2 / wang3 / wang4); anything else
// keeps the one-kernel-per-op path (nas.cu).
#pragma once

#include "common.cuh"
#include "tc_conv.cuh"

namespace hn {

#ifndef HN_TAIL_UNROLL_LIMIT
#define HN_TAIL_UNROLL_LIMIT 0
#endif
constexpr int kTailMaxOps = 24;
constexpr int kTailMaxWG = 6;    // 768 threads: 85 registers per thread
constexpr int kTailBars = 8;     // mbarrier slots per kind
enum : int { TAIL_PW = 1, TAIL_DW = 2, TAIL_POOL = 3 };

struct TailOp {
  int kind;
  int shape;                       // PW: 0..4 = (cin, cout, pixels) below; DW / POOL: 0..4 = (C, hout, stride) below
  int kernel, relu;
  int src_off, dst_off, res_off;   // byte offsets inside the warpgroup's buffer region (res: -1 = none)
  int w_off, b_off;                // byte offsets from the aligned shared-memory base (weight blob)
  int parity;                      // PW: the output is written in / DW, POOL (stride 2): the input is read from the "parity layout" below
};

struct TailParams {
  const uint16_t* in;     // [n][in_planes][in_pix][8] channel-planar fp16 (input of ops[0]): one bulk copy per patch
  uint16_t* out;          // output of ops[n_ops - 1]: channel-planar like the input (out_planar: another tail launch or the head
                          // GEMM, whose weight K order is permuted to match, reads it) or [n][out_pix][out_planes * 8] NHWC
  const uint4* blob;      // weight image in global memory (copied once per CTA)
  int blob_off, blob_bytes;
  int n, n_ops;
  int wg_stride;          // bytes of one warpgroup's buffer region (region w starts at w * wg_stride)
  int bar_off;            // 2 x kTailMaxWG mbarriers ("accumulators complete", "input landed") + tensor-memory slot
  int ones_off;           // constant A tile [128 rows][K = 16]: columns 0, 1 = 1.0 (its second K plane = 2 KB of zeros), then 16 B of -inf
  int eye_off;            // constant B tile: 16 x 16 identity
  int in_off, in_bytes;   // the patch's input region / bytes
  int out_off, out_pix, out_planes_log2, out_planar;
  int prefetch_after;     // index of the last op that touches the input region: the NEXT patch's input is requested right
                          // behind it and lands while the remaining ops run (-1: the region is busy to the end)
  int op_base, launch_id; // index of ops[0] in the program / of this launch in the plan (diagnostics)
  TailOp ops[kTailMaxOps];
};

#ifdef HN_TAIL_TRACE
// Diagnostic build only (-DHN_TAIL_TRACE): cycles thread 0 of CTA 0 spends per op ([program op index]; PW: [64 + op] up to
// "accumulators complete"), load [32 + launch], store [40 + launch], total [48 + launch], patches [56 + launch]
__device__ unsigned long long hn_tail_trace[128];
#define HN_TAIL_T(var) const long long var = clock64()
#define HN_TAIL_ACC(slot, t0) do { if (blockIdx.x == 0 && threadIdx.x == 0) hn_tail_trace[slot] += static_cast<unsigned long long>(clock64() - (t0)); } while (0)
#else
#define HN_TAIL_T(var) do { } while (0)
#define HN_TAIL_ACC(slot, t0) do { } while (0)
#endif

// A map whose only reader is a stride-2 depthwise conv / max-pool is laid out by its producer so that the taps of
// consecutive output columns are consecutive 16-byte slots (plain rows give a 32-byte lane stride = two shared-memory
// wavefronts per quarter warp): a row holds its even columns, then its odd columns. 16-wide rows rotate the odd half by four
// slots so that the producer's eight consecutive pixels still hit eight different bank groups; 8-wide rows swap the halves
// on every second row pair so that two strips of one quarter warp (rows 2 apart) use different halves.
template <int W>
__device__ __forceinline__ int tail_parity_slot(int y, int x) {
  static_assert(W == 16 || W == 8, "maps read at stride 2 behind the front stage");
  if constexpr (W == 16) return y * 16 + ((x & 1) ? 8 + (((x >> 1) + 4) & 7) : (x >> 1));
  else return y * 8 + ((((x & 1) ^ (y >> 1)) & 1) << 2) + (x >> 1);
}

__device__ __forceinline__ void tail_wg_sync(int wg) { asm volatile("bar.sync %0, 128;" ::"r"(wg + 1) : "memory"); }

// ---- depthwise conv / max-pool of one patch by the 128 threads of a warpgroup -------------------------------------------
template <int K, int S, int C, int HOUT, bool POOL, bool PAR = false>
__device__ __forceinline__ void tail_dw(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, const uint8_t* __restrict__ s_w /*[K * K][C] fp16*/,
                                        const uint8_t* __restrict__ s_b /*[C] fp16*/, const uint8_t* __restrict__ s_pad /*16 B of padding value*/,
                                        int relu, int t) {
  constexpr int HIN = HOUT * S, PLANES = C / 8, PAD = K >> 1;
  constexpr int SH = PLANES * HOUT * HOUT / 128;
  static_assert(SH >= 1 && SH * 128 == PLANES * HOUT * HOUT && HOUT % SH == 0, "one item per thread");
  static_assert(!PAR || S == 2, "the parity layout serves stride-2 readers");
  constexpr int STRIPS = HOUT / SH, NR = (SH - 1) * S + K;
  const int ox = t % HOUT, ys = (t / HOUT) % STRIPS, plane = t / (HOUT * STRIPS);
  const uint8_t* map = src + plane * (HIN * HIN * 16);
  constexpr uint32_t kNinf = 0xFC00FC00u;
  __half2 acc[SH][4];
  if constexpr (POOL) {
#pragma unroll
    for (int j = 0; j < SH; ++j)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[j][c] = *reinterpret_cast<const __half2*>(&kNinf);
  } else {
    const uint4 b = *reinterpret_cast<const uint4*>(s_b + plane * 16);
#pragma unroll
    for (int j = 0; j < SH; ++j) {
      acc[j][0] = *reinterpret_cast<const __half2*>(&b.x); acc[j][1] = *reinterpret_cast<const __half2*>(&b.y);
      acc[j][2] = *reinterpret_cast<const __half2*>(&b.z); acc[j][3] = *reinterpret_cast<const __half2*>(&b.w);
    }
  }
  const int iy0 = ys * SH * S - PAD;
  // small bodies are unrolled over kx (the loads of the next column overlap this column's arithmetic); the 5x5 stride-1
  // strip of 8 rows stays rolled: its body alone is ~220 instructions and the kernel's hot code must stay i-cache sized
  constexpr int UNR = (SH * K * K * 4 <= HN_TAIL_UNROLL_LIMIT) ? K : 1;
#pragma unroll UNR
  for (int kx = 0; kx < K; ++kx) {
    const int ix = ox * S + kx - PAD;
    const bool x_ok = ix >= 0 && ix < HIN;
    uint4 wk[K];
    if constexpr (!POOL) {
#pragma unroll
      for (int ky = 0; ky < K; ++ky) wk[ky] = *reinterpret_cast<const uint4*>(s_w + ((ky * K + kx) * C + plane * 8) * 2);
    }
    // out-of-image taps read a padding vector (one select on the address; no predicated load, no register zeroing); its bank
    // group is one the in-image lanes of the quarter warp cannot use (they end at group 7 on the left border, start at 0 on the right)
    const uint8_t* pad = s_pad + ((S == 1 && kx < PAD) ? 112 : 0);
    int xs = ix;
    if constexpr (PAR && HIN == 16) xs = (ix & 1) ? 8 + (((ix >> 1) + 4) & 7) : (ix >> 1);
    const uint8_t* col = map + xs * 16 + iy0 * (HIN * 16);
#pragma unroll
    for (int r = 0; r < NR; ++r) {
      const bool ok = x_ok && static_cast<unsigned>(iy0 + r) < static_cast<unsigned>(HIN);
      const uint8_t* ptr = col + r * (HIN * 16);
      if constexpr (PAR && HIN == 8) ptr = map + tail_parity_slot<8>(iy0 + r, ix) * 16;
      const uint4 xv = *reinterpret_cast<const uint4*>(ok ? ptr : pad);
      const __half2 x[4] = {*reinterpret_cast<const __half2*>(&xv.x), *reinterpret_cast<const __half2*>(&xv.y),
                            *reinterpret_cast<const __half2*>(&xv.z), *reinterpret_cast<const __half2*>(&xv.w)};
#pragma unroll
      for (int j = 0; j < SH; ++j) {
        const int ky = r - j * S;            // compile-time after unrolling
        if (ky >= 0 && ky < K) {
          if constexpr (POOL) {
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[j][c] = __hmax2_nan(acc[j][c], x[c]);
          } else {
            const __half2 w[4] = {*reinterpret_cast<const __half2*>(&wk[ky].x), *reinterpret_cast<const __half2*>(&wk[ky].y),
                                  *reinterpret_cast<const __half2*>(&wk[ky].z), *reinterpret_cast<const __half2*>(&wk[ky].w)};
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[j][c] = __hfma2(x[c], w[c], acc[j][c]);
          }
        }
      }
    }
  }
  uint8_t* optr = dst + plane * (HOUT * HOUT * 16) + ((ys * SH) * HOUT + ox) * 16;
  const __half2 hzero = __float2half2_rn(0.f);
#pragma unroll
  for (int j = 0; j < SH; ++j) {
    if (!POOL && relu) {
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[j][c] = __hmax2(acc[j][c], hzero);
    }
    *reinterpret_cast<uint4*>(optr + j * (HOUT * 16)) =
        make_uint4(*reinterpret_cast<const uint32_t*>(&acc[j][0]), *reinterpret_cast<const uint32_t*>(&acc[j][1]),
                   *reinterpret_cast<const uint32_t*>(&acc[j][2]), *reinterpret_cast<const uint32_t*>(&acc[j][3]));
  }
}

// {lo, hi} -> two fp16 values saturated to the largest finite value, one instruction
__device__ __forceinline__ uint32_t tail_pack_sat(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// ---- pointwise conv of one patch: MMAs issued by one lane of the warpgroup's first warp, epilogue by its four warps ------
// COLS = the warpgroup's tensor-memory columns (128 with up to four warpgroups per CTA, 64 with five or six): an op whose
// accumulators need more (C_out = 128) runs as two column passes of N = 64, one after the other.
// RESW > 0: a second input tensor of RESW channels with its own weights (a folded block: y = relu(W a + W1 x + b), nas.cu);
// RESW == 0 and res_off >= 0: a plain residual, added through 16 x 16 identity slices.
template <int CIN, int COUT, int ROWS, int COLS, int STEP_MAX, int RESW = 0>
__device__ __forceinline__ void tail_pw(uint8_t* __restrict__ buf, uint32_t buf_addr, const uint8_t* __restrict__ sm, uint32_t base,
                                        const TailOp& o, int ones_off, int eye_off, uint32_t tmem_wg, uint32_t bar, uint32_t& phase, int wg,
                                        int q, int lane, int trace_op) {
  HN_TAIL_T(t_pw);
  constexpr int TILES = (ROWS + kTileM - 1) / kTileM;
  constexpr uint32_t PITCH = ROWS * 16;                  // plane pitch of the (equal-sized) source / destination maps
  constexpr int NPASS = (TILES * COUT + COLS - 1) / COLS;
  constexpr int NP = COUT / NPASS;                       // output channels per pass = N of its MMAs
  static_assert(NP * NPASS == COUT && TILES * NP <= COLS && NP % 32 == 0 && CIN % 16 == 0, "accumulators of one pass fit the warpgroup's columns");
  uint8_t* dstp = buf + o.dst_off;
  const int relu = o.relu;
#pragma unroll
  for (int np = 0; np < NPASS; ++np) {
    if (np > 0) {                                         // every warp has drained the previous pass from tensor memory
      tc_fence_before();
      tail_wg_sync(wg);
    }
    if (q == 0) {
      tc_fence_after();
      if (elect_one()) {
        constexpr uint32_t a_hi = noswizzle_desc_hi(128);
        constexpr int KP = CIN + 16 + RESW;                // K of the weight image: [W | bias hi, lo, 0... | W1]
        constexpr uint32_t b_hi = noswizzle_desc_hi(KP * 16);
        constexpr uint32_t idesc = make_idesc_f16(kTileM, NP, 0);
        const uint32_t a_lo0 = noswizzle_desc_lo(buf_addr + o.src_off, PITCH);
        // weight image rows [np * NP, (np + 1) * NP): 8-row groups are KP * 16 bytes apart
        const uint32_t b_lo0 = noswizzle_desc_lo(base + o.w_off + np * (NP / 8) * (KP * 16), 128);
        const uint32_t ones_lo = noswizzle_desc_lo(base + ones_off, 2048);
#pragma unroll
        for (int t = 0; t < TILES; ++t) {
#pragma unroll
          for (int k = 0; k < CIN / 16; ++k)
            umma_f16_w(tmem_wg + t * NP, a_lo0 + t * (2048u >> 4) + k * ((2u * PITCH) >> 4), a_hi, b_lo0 + k * 16u, b_hi, idesc, k != 0);
          // + bias: a K step of the constant "ones" tile against the weight image's last 16 K columns (bias as fp16 hi + lo)
          umma_f16_w(tmem_wg + t * NP, ones_lo, a_hi, b_lo0 + (CIN / 16) * 16u, b_hi, idesc, 1u);
          if constexpr (RESW > 0) {
            // + W1 x: K steps over the second input (same pixel pitch) against the image's last RESW K columns
            const uint32_t x_lo0 = noswizzle_desc_lo(buf_addr + o.res_off, PITCH);
#pragma unroll
            for (int k = 0; k < RESW / 16; ++k)
              umma_f16_w(tmem_wg + t * NP, x_lo0 + t * (2048u >> 4) + k * ((2u * PITCH) >> 4), a_hi, b_lo0 + (CIN / 16 + 1 + k) * 16u, b_hi, idesc, 1u);
          }
        }
        if (RESW == 0 && o.res_off >= 0) {
          // + residual: 16-channel slices of the block input against a 16 x 16 identity (exact in the fp32 accumulator)
          constexpr uint32_t e_hi = noswizzle_desc_hi(256);
          constexpr uint32_t idesc16 = make_idesc_f16(kTileM, 16, 0);
          const uint32_t r_lo0 = noswizzle_desc_lo(buf_addr + o.res_off + np * (NP / 8) * PITCH, PITCH);
          const uint32_t e_lo = noswizzle_desc_lo(base + eye_off, 128);
#pragma unroll
          for (int t = 0; t < TILES; ++t) {
#pragma unroll
            for (int k = 0; k < NP / 16; ++k)
              umma_f16_w(tmem_wg + t * NP + k * 16, r_lo0 + t * (2048u >> 4) + k * ((2u * PITCH) >> 4), a_hi, e_lo, e_hi, idesc16, 1u);
          }
        }
        umma_commit(bar);
      }
      __syncwarp();
    }
    mbar_wait(bar, phase);
    phase ^= 1u;
    tc_fence_after();
    if (np == 0) HN_TAIL_ACC(64 + trace_op, t_pw);
    // epilogue: accumulator (bias and residual already inside) -> [ReLU] -> fp16 -> planar destination, up to two 32-column
    // loads in flight
    constexpr int CH = NP / 32;                            // 32-column chunks per tile
    constexpr int NCH = TILES * CH;
    static_assert(NCH == 1 || NCH % 2 == 0, "chunks are processed in pairs");
    constexpr int STEP = (NCH >= 2 && STEP_MAX >= 2) ? 2 : 1;
#pragma unroll
    for (int c = 0; c < NCH; c += STEP) {
      if ((TILES == 1 ? 0 : (c / CH) * kTileM) + q * 32 < ROWS) {   // warp-uniform (two tiles only with full maps)
        uint32_t r[STEP][32];
#pragma unroll
        for (int u = 0; u < STEP; ++u) {
          const int tt = (c + u) / CH, c0 = ((c + u) % CH) * 32;
          tmem_ld32(tmem_wg + (static_cast<uint32_t>(q * 32) << 16) + tt * NP + c0, r[u]);
        }
        tmem_ld_wait();
#pragma unroll
        for (int u = 0; u < STEP; ++u) {
          const int tt = (c + u) / CH, c0 = np * NP + ((c + u) % CH) * 32;
          const int row = tt * kTileM + q * 32 + lane;
          int slot = row;
          if constexpr (ROWS == 256) { if (o.parity) slot = tail_parity_slot<16>(row >> 4, row & 15); }
          if constexpr (ROWS == 64) { if (o.parity) slot = tail_parity_slot<8>(row >> 3, row & 7); }
          if (row < ROWS) {
#pragma unroll
            for (int h = 0; h < 4; ++h) {
              const uint32_t poff = static_cast<uint32_t>(c0 / 8 + h) * PITCH + slot * 16;
              const float* v = reinterpret_cast<const float*>(&r[u][8 * h]);
              uint4 ov;
              if (relu)
                ov = make_uint4(pack16_relu(v[0], v[1], 0), pack16_relu(v[2], v[3], 0), pack16_relu(v[4], v[5], 0), pack16_relu(v[6], v[7], 0));
              else
                ov = make_uint4(tail_pack_sat(v[0], v[1]), tail_pack_sat(v[2], v[3]), tail_pack_sat(v[4], v[5]), tail_pack_sat(v[6], v[7]));
              *reinterpret_cast<uint4*>(dstp + poff) = ov;
            }
          }
        }
      }
    }
  }
}

template <int NWG>
__global__ void __launch_bounds__(NWG * 128, 1) nas_tail_kernel(const __grid_constant__ TailParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (base - raw_addr);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int wg = warp >> 2, q = warp & 3, t = threadIdx.x & 127;
  const uint32_t bar0 = base + p.bar_off;
  const uint32_t tmem_slot = bar0 + 16 * kTailBars;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(sm + p.bar_off + 16 * kTailBars);

  if (warp == 0) {
    if (lane == 0) {
      for (int i = 0; i < NWG; ++i) {
        mbar_init(bar0 + 8 * i, 1);
        mbar_init(bar0 + 8 * (kTailBars + i), 1);
      }
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  {
    uint4* dst = reinterpret_cast<uint4*>(sm + p.blob_off);
    for (int i = threadIdx.x; i < p.blob_bytes / 16; i += NWG * 128) dst[i] = __ldg(p.blob + i);
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  constexpr int COLS = NWG <= 4 ? 128 : 64;            // tensor-memory columns per warpgroup
  constexpr int STEPM = NWG <= 4 ? 2 : 1;              // 32-column accumulator loads in flight (register budget)
  const uint32_t tmem_wg = *tmem_slot_ptr + wg * COLS;
  const uint32_t bar = bar0 + 8 * wg;
  const uint32_t bar_ld = bar0 + 8 * (kTailBars + wg);
  uint32_t phase = 0, phase_ld = 0;
  uint8_t* buf = sm + wg * p.wg_stride;
  const uint32_t buf_addr = base + wg * p.wg_stride;
  const size_t out_patch_bytes = static_cast<size_t>(p.out_pix) << (4 + p.out_planes_log2);
  const int stride = gridDim.x * NWG;
  const int pf = (p.prefetch_after >= 0 && p.prefetch_after < p.n_ops - 1) ? p.prefetch_after : -1;
  // one thread of the warpgroup requests a patch's input: ONE bulk copy (the global layout is the shared-memory layout)
  auto request = [&](int patch) {
    mbar_arrive_expect_tx(bar_ld, static_cast<uint32_t>(p.in_bytes));
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(buf_addr + p.in_off),
                 "l"(reinterpret_cast<const uint8_t*>(p.in) + static_cast<size_t>(patch) * p.in_bytes), "r"(static_cast<uint32_t>(p.in_bytes)), "r"(bar_ld)
                 : "memory");
  };

  HN_TAIL_T(t_total);
  int patch = blockIdx.x * NWG + wg;
  if (t == 0 && patch < p.n) request(patch);
  for (; patch < p.n; patch += stride) {
    HN_TAIL_T(t_load);
    if (t == 0) bulk_wait_read<0>();   // the previous patch's output store has left shared memory
    mbar_wait(bar_ld, phase_ld);
    phase_ld ^= 1u;
    tail_wg_sync(wg);
    HN_TAIL_ACC(32 + p.launch_id, t_load);

    for (int oi = 0; oi < p.n_ops; ++oi) {
      const TailOp& o = p.ops[oi];
      HN_TAIL_T(t_op);
      if (o.kind == TAIL_PW) {
#define HN_TAIL_PW(CI, CO, R, RW) tail_pw<CI, CO, R, COLS, STEPM, RW>(buf, buf_addr, sm, base, o, p.ones_off, p.eye_off, tmem_wg, bar, phase, wg, q, lane, p.op_base + oi)
        // five or six warpgroups only fit when no 16 x 16 map is part of the run (8 KB regions): those shapes are not compiled in
        if constexpr (NWG <= 4) {
          if (o.shape == 0) HN_TAIL_PW(32, 32, 256, 0);
          if (o.shape == 5) HN_TAIL_PW(32, 32, 256, 32);
        }
        switch (o.shape) {        // (cin, weighted second-input channels, cout, pixels): tail_pw_shape in nas.cu
          case 0: case 5: break;
          case 1: HN_TAIL_PW(32, 64, 64, 0); break;
          case 2: HN_TAIL_PW(64, 64, 64, 0); break;
          case 3: HN_TAIL_PW(64, 128, 16, 0); break;
          case 4: HN_TAIL_PW(128, 128, 16, 0); break;
          case 6: HN_TAIL_PW(64, 64, 64, 32); break;
          case 7: HN_TAIL_PW(64, 64, 64, 64); break;
          default: HN_TAIL_PW(128, 128, 16, 64); break;
        }
#undef HN_TAIL_PW
      } else if (o.kind == TAIL_DW) {
        const uint8_t* s = buf + o.src_off;
        uint8_t* d = buf + o.dst_off;
        const uint8_t* w = sm + o.w_off;
        const uint8_t* b = sm + o.b_off;
        const uint8_t* pad0 = sm + p.ones_off + 2048;   // zeros
#define HN_TAIL_DW(K_, S_, C_, H_) tail_dw<K_, S_, C_, H_, false>(s, d, w, b, pad0, o.relu, t)
#define HN_TAIL_DW2(K_, C_, H_) do { if (o.parity) tail_dw<K_, 2, C_, H_, false, true>(s, d, w, b, pad0, o.relu, t); else HN_TAIL_DW(K_, 2, C_, H_); } while (0)
        if constexpr (NWG <= 4) {                       // 16 x 16 inputs: never with five or six warpgroups (see above)
          if (o.shape == 0) { if (o.kernel == 3) HN_TAIL_DW(3, 1, 32, 16); else HN_TAIL_DW(5, 1, 32, 16); }
          if (o.shape == 1) { if (o.kernel == 3) HN_TAIL_DW2(3, 32, 8); else HN_TAIL_DW2(5, 32, 8); }
        }
        if (o.kernel == 3) {
          switch (o.shape) {
            case 0: case 1: break;
            case 2: HN_TAIL_DW(3, 1, 64, 8); break;
            case 3: HN_TAIL_DW2(3, 64, 4); break;
            default: HN_TAIL_DW(3, 1, 128, 4); break;
          }
        } else {
          switch (o.shape) {
            case 0: case 1: break;
            case 2: HN_TAIL_DW(5, 1, 64, 8); break;
            case 3: HN_TAIL_DW2(5, 64, 4); break;
            default: HN_TAIL_DW(5, 1, 128, 4); break;
          }
        }
#undef HN_TAIL_DW2
#undef HN_TAIL_DW
      } else {
        const uint8_t* padn = sm + p.ones_off + 4096;   // -inf
        const uint8_t* s = buf + o.src_off;
        uint8_t* d = buf + o.dst_off;
        if (o.shape == 1) {
          if constexpr (NWG <= 4) {
            if (o.parity) tail_dw<3, 2, 32, 8, true, true>(s, d, nullptr, nullptr, padn, 0, t);
            else tail_dw<3, 2, 32, 8, true>(s, d, nullptr, nullptr, padn, 0, t);
          }
        } else {
          if (o.parity) tail_dw<3, 2, 64, 4, true, true>(s, d, nullptr, nullptr, padn, 0, t);
          else tail_dw<3, 2, 64, 4, true>(s, d, nullptr, nullptr, padn, 0, t);
        }
      }
      // the next op reads this one's output through the other proxy (generic <-> tensor core) and may overwrite its
      // accumulators / source buffer
      tc_fence_before();
      fence_proxy_async_smem();
      tail_wg_sync(wg);
      if (oi == pf && t == 0 && patch + stride < p.n) request(patch + stride);
      HN_TAIL_ACC(p.op_base + oi, t_op);
    }

    HN_TAIL_T(t_store);
    if (p.out_planar) {
      // one bulk store (every thread fenced its writes towards the async proxy behind the last op)
      if (t == 0) {
        bulk_store(reinterpret_cast<uint8_t*>(p.out) + static_cast<size_t>(patch) * out_patch_bytes, buf_addr + p.out_off,
                   static_cast<uint32_t>(out_patch_bytes));
        bulk_commit();
      }
    } else {
      // channel-planar shared memory -> NHWC global in 16-byte chunks: chunk i = (pixel block, plane, pixel % 8), so 8
      // consecutive lanes read 128 contiguous bytes of one plane while the warp writes whole lines of the NHWC tensor
      uint8_t* dst = reinterpret_cast<uint8_t*>(p.out) + static_cast<size_t>(patch) * out_patch_bytes;
      const int pl2 = p.out_planes_log2;
      const uint32_t pitch = static_cast<uint32_t>(p.out_pix) * 16;
      const uint8_t* s0 = buf + p.out_off;
      const int chunks = p.out_pix << pl2;
      for (int i = t; i < chunks; i += 128) {
        const int blk = i >> (3 + pl2), rem = i & ((8 << pl2) - 1);
        const int plane = rem >> 3, pixel = blk * 8 + (rem & 7);
        *reinterpret_cast<uint4*>(dst + ((static_cast<size_t>(pixel) << pl2) + plane) * 16) =
            *reinterpret_cast<const uint4*>(s0 + plane * pitch + pixel * 16);
      }
      tail_wg_sync(wg);   // the output region may be overwritten by the next patch
    }
    if (pf < 0 && t == 0 && patch + stride < p.n) {
      bulk_wait_read<0>();             // the output may share the input region
      request(patch + stride);
    }
    HN_TAIL_ACC(40 + p.launch_id, t_store);
#ifdef HN_TAIL_TRACE
    if (blockIdx.x == 0 && threadIdx.x == 0) hn_tail_trace[56 + p.launch_id] += 1;
#endif
  }
  HN_TAIL_ACC(48 + p.launch_id, t_total);

  if (t == 0) bulk_wait_all<0>();      // output stores still read this CTA's shared memory
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(*tmem_slot_ptr, 512);
  }
}

}  // namespace hn
