// C ABI for the distance / hardest-in-batch / matching path: operand packing, the fused tcgen05
// distance kernels (tc_dist.cuh), fp32 re-ranking of shortlisted candidates and the small finalisers.
#include <algorithm>
#include <cmath>
#include <type_traits>
#include <vector>

#include "host_common.h"
#include "tc_dist.cuh"
#include "tc_dist_pair.cuh"

namespace hn {

constexpr float kOperandScale = 256.0f;  // descriptors are unit vectors: x256 keeps the fp16 hi/lo split clear of subnormals
constexpr float kDotScale = 1.0f / (kOperandScale * kOperandScale);
// |fp16-operand dot - exact dot| <= 2^-10 for rows of norm <= 1 (L2-normalised descriptors, the only input matching is defined
// for: FDLNet-master/utils/math_utils.py:15-18 clamps 2 - 2ab to [1e-8, 4]). In the GEMM's scaled units, the re-rank keeps 4x
// that bound as the margin of its candidate threshold and the mutual verification 2x as the margin of its cell test.
// e4m3 rows (packed as exact e4m3 x * 2^8, kind::f8f6f4 GEMM): every product is exact, so the dot error is the tensor core's
// accumulation alone, which PTX does not specify. The bound relied on, and its assumption: each MMA (K = 32) adds its 32
// products to the fp32 accumulator with an error of at most 2^-18 times the largest magnitude involved (a product or the
// running sum) per term, i.e. it keeps at least 18 bits below the leading bit of the aligned sum (true fp32 accumulation keeps
// 23; with scaled operands every partial sum is a multiple of 2^-2 below 2^17, so fp32 accumulation is exact). Rows rounded to
// e4m3 have norm <= (1 + 2^-4) + sqrt(128) * 2^-10 < 1.074 (relative rounding 2^-4 plus the subnormal spacing), so every
// product and partial sum is <= 1.074^2 < 1.16 and the error of a 128-term dot is <= 4 MMAs * 33 terms * 2^-18 * 1.16 < 5.9e-4
// < 2^-10. The fp16 bound holds, and the same margins keep the same factor of two. tests/test_matching_fp8_gpu.py checks the
// bound (kF8DotBound below, in unscaled units) against float64 cell maxima of adversarial e4m3 rows.
constexpr float kF8DotBound = 5.9e-4f;
static_assert(kF8DotBound <= 1.0f / 1024.0f, "the fp8 GEMM's error must stay within the bound the margins are made of");
constexpr float kRerankMargin = 4.0f * (1.0f / 1024.0f) / kDotScale;
constexpr float kVerifyMargin = 2.0f * (1.0f / 1024.0f) / kDotScale;

static inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

// Descriptor rows of the matching kernels are fp32, fp16 or bf16 (T = float, __half, __nv_bfloat16). A lane reads elements
// 4 * lane ... 4 * lane + 3 of a row as fp32: one 16-byte load for fp32 rows, one 8-byte load for 16-bit rows, converted on the
// spot. Every fp16 / bf16 value is an fp32 value, so a kernel on 16-bit rows computes exactly what it computes on x.float().
__device__ __forceinline__ float4 row4_from_bits(uint2 v, __half) {
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&v.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ float4 row4_from_bits(uint2 v, __nv_bfloat16) {
  const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v.x));
  const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
// e4m3 rows (HN_F8E4M3): one 4-byte load per lane, four exact e4m3 -> fp16 -> fp32 conversions.
__device__ __forceinline__ float4 row4_from_bits(uint32_t v, __nv_fp8_e4m3) {
  const __half2_raw a = __nv_cvt_fp8x2_to_halfraw2(static_cast<__nv_fp8x2_storage_t>(v & 0xffffu), __NV_E4M3);
  const __half2_raw b = __nv_cvt_fp8x2_to_halfraw2(static_cast<__nv_fp8x2_storage_t>(v >> 16), __NV_E4M3);
  const float2 fa = __half22float2(__half2(a)), fb = __half22float2(__half2(b));
  return make_float4(fa.x, fa.y, fb.x, fb.y);
}
__device__ __forceinline__ float4 ld_row4(const float* row, int lane) { return reinterpret_cast<const float4*>(row)[lane]; }
__device__ __forceinline__ float4 ld_row4(const __nv_fp8_e4m3* row, int lane) {
  return row4_from_bits(reinterpret_cast<const uint32_t*>(row)[lane], __nv_fp8_e4m3{});
}
__device__ __forceinline__ float4 ldg_row4(const __nv_fp8_e4m3* row, int lane) {
  return row4_from_bits(__ldg(reinterpret_cast<const unsigned int*>(row) + lane), __nv_fp8_e4m3{});
}
__device__ __forceinline__ float4 ldg_row4(const float* row, int lane) { return __ldg(reinterpret_cast<const float4*>(row) + lane); }
template <typename T>
__device__ __forceinline__ float4 ld_row4(const T* row, int lane) { return row4_from_bits(reinterpret_cast<const uint2*>(row)[lane], T{}); }
template <typename T>
__device__ __forceinline__ float4 ldg_row4(const T* row, int lane) { return row4_from_bits(__ldg(reinterpret_cast<const uint2*>(row) + lane), T{}); }

// [n,128] rows -> 16-bit K-major operand rows. split == 0: [hi] (K=128). split == 1 (fp32 rows only): K=384,
// order 0 = [hi, hi, lo] (row side), order 1 = [hi, lo, hi] (column side), so that the GEMM accumulates
// hi*hi + hi*lo + lo*hi. Also emits |x|^2 (torch.sum(x*x, dim=1), hardnet/Losses.py:8-9). 16-bit rows are widened to fp32
// first, so their operand rows equal those of x.float() bit for bit.
template <typename T>
__global__ void pack_desc_kernel(const T* __restrict__ x, long long n, uint16_t* __restrict__ out, int split, int order,
                                 float* __restrict__ norm) {
  const long long row = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n) return;
  const float4 v = ld_row4(x + row * 128, lane);
  const float f[4] = {v.x, v.y, v.z, v.w};
  float ss = (f[0] * f[0] + f[1] * f[1]) + (f[2] * f[2] + f[3] * f[3]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if (norm && lane == 0) norm[row] = ss;
  uint16_t hi[4], lo[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float s = f[j] * kOperandScale;
    const __half h = __float2half_rn(s);
    const __half l = __float2half_rn(s - __half2float(h));
    hi[j] = __half_as_ushort(h);
    lo[j] = __half_as_ushort(l);
  }
  const int K = split ? 384 : 128;
  uint16_t* dst = out + row * K + lane * 4;
  const uint2 H = make_uint2(hi[0] | (uint32_t(hi[1]) << 16), hi[2] | (uint32_t(hi[3]) << 16));
  const uint2 L = make_uint2(lo[0] | (uint32_t(lo[1]) << 16), lo[2] | (uint32_t(lo[3]) << 16));
  *reinterpret_cast<uint2*>(dst) = H;
  if (split) {
    *reinterpret_cast<uint2*>(dst + 128) = order == 0 ? H : L;
    *reinterpret_cast<uint2*>(dst + 256) = order == 0 ? L : H;
  }
}

// [n,128] e4m3 rows -> e4m3 operand rows x * 2^8 (exact for |x| <= 1, see the margin comment), one 4-byte word per lane.
__global__ void pack_desc_f8_kernel(const __nv_fp8_e4m3* __restrict__ x, long long n, uint32_t* __restrict__ out) {
  const long long row = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n) return;
  const float4 v = ld_row4(x + row * 128, lane);
  out[row * 32 + lane] = pack_e4m3x4(v.x * kOperandScale, v.y * kOperandScale, v.z * kOperandScale, v.w * kOperandScale);
}

// Push all-gather over NVSwitch multicast: a rank packs its shard and writes BOTH forms (fp16 operand rows for the GEMM, fp32
// rows for the exact re-rank) to multicast addresses (multimem.st): the switch replicates every 16-byte store into the
// symmetric buffer of every GPU of the group, so after one cross-GPU barrier each GPU holds the whole gallery without a
// gather kernel, a copy engine or a second pass over the data. Half a warp per row: a lane owns 8 consecutive floats.
__global__ void pack_desc_multicast_kernel(const float* __restrict__ x, long long n, uint16_t* __restrict__ mc16,
                                           float* __restrict__ mc32) {
  const long long gid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long row = gid >> 4;
  const int l = static_cast<int>(gid & 15);
  if (row >= n) return;
  const float4 a = reinterpret_cast<const float4*>(x + row * 128)[2 * l];
  const float4 b = reinterpret_cast<const float4*>(x + row * 128)[2 * l + 1];
  const float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  uint32_t h[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const __half2 v = __floats2half2_rn(f[2 * j] * kOperandScale, f[2 * j + 1] * kOperandScale);
    h[j] = *reinterpret_cast<const uint32_t*>(&v);
  }
  if (mc16 != nullptr)
    asm volatile("multimem.st.weak.global.v4.f16x2 [%0], {%1, %2, %3, %4};" ::"l"(mc16 + row * 128 + l * 8), "r"(h[0]), "r"(h[1]),
                 "r"(h[2]), "r"(h[3])
                 : "memory");
  if (mc32 != nullptr) {
    asm volatile("multimem.st.weak.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc32 + row * 128 + l * 8), "f"(a.x), "f"(a.y),
                 "f"(a.z), "f"(a.w)
                 : "memory");
    asm volatile("multimem.st.weak.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc32 + row * 128 + l * 8 + 4), "f"(b.x), "f"(b.y),
                 "f"(b.z), "f"(b.w)
                 : "memory");
  }
  // no per-thread fence: the stores are complete when the kernel retires, and the cross-GPU barrier that follows on the same
  // stream publishes them (release / acquire at system scope); a __threadfence_system() here cost 0.1 ms per 24 MiB
}

__global__ void unpack_min_kernel(const unsigned long long* __restrict__ pack, long long n, float* __restrict__ val,
                                  int* __restrict__ arg) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long pk = pack[i];
  if (val) val[i] = __uint_as_float(static_cast<unsigned int>(pk >> 32));
  if (arg) arg[i] = static_cast<int>(pk & 0xffffffffu);
}

// mean(clamp(margin + pos - min_neg, 0)) with min_neg = min(row_min, col_min) — hardnet/Losses.py:105-108,
// 142-143,153. One block, fixed summation order -> deterministic.
__global__ void loss_finalize_kernel(const float* __restrict__ pos, const unsigned long long* __restrict__ row_pack,
                                     const unsigned long long* __restrict__ col_pack, long long n, float margin,
                                     float* __restrict__ out) {
  __shared__ float red[32];
  float acc = 0.f;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) {
    float mn = __uint_as_float(static_cast<unsigned int>(row_pack[i] >> 32));
    if (col_pack) mn = fminf(mn, __uint_as_float(static_cast<unsigned int>(col_pack[i] >> 32)));
    acc += fmaxf(margin + pos[i] - mn, 0.f);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (threadIdx.x == 0) out[0] = v / static_cast<float>(n);
  }
}

// Top-2 of one query row: distances d1 <= d2 and their gallery columns (0x7fffffff: fewer columns than that).
struct Top2 {
  float d1, d2;
  int i1, i2;
};

// Exact fp32 distances of the kChunk columns col0 ... col0 + 7 of g to one query row, for a warp whose lane holds elements
// 4 * lane ... 4 * lane + 3 of that row in qv: lane r < kChunk (and every lane r + 8 j) returns the distance of column col0 + r,
// for r < left (the columns that exist). The warp reads a gallery row as ONE coalesced 512 B read (lane = float4 index) and
// finishes the 128-term dot with a butterfly, so every lane holds the same dot products. Per-lane row reads (one lane per
// candidate) cost 32 L1 wavefronts per row instead of 4. rerank_row and rerank_topk_row both evaluate chunks here, so their
// distances agree bit for bit.
template <typename T>
__device__ __forceinline__ float chunk_distance(float4 qv, const T* g, long long col0, long long left, int lane) {
  float part[kChunk];
#pragma unroll
  for (int r = 0; r < kChunk; ++r) {
    part[r] = 0.f;
    if (r < left) {
      const float4 gv = ldg_row4(g + (col0 + r) * 128, lane);
      part[r] = fmaf(qv.x, gv.x, fmaf(qv.y, gv.y, fmaf(qv.z, gv.z, qv.w * gv.w)));
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int r = 0; r < kChunk; ++r) part[r] += __shfl_xor_sync(0xffffffffu, part[r], o);
  }
  // The eight distances are taken by eight lanes, one sqrtf each, and shuffled to the warp by the caller (every lane holds the
  // same eight dot products). Eight unrolled sqrtf per lane are eight slow-path calls, across which the gallery pointer and size
  // stay live: that made ptxas spill.
  float mine = part[0];   // part[lane & 7] without a local-memory array access
#pragma unroll
  for (int r = 1; r < kChunk; ++r) mine = (lane & (kChunk - 1)) == r ? part[r] : mine;
  return sqrtf(fminf(fmaxf(2.0f - 2.0f * mine, 1e-8f), 4.0f));
}

// Exact fp32 re-rank of the shortlisted chunks of one query row: one warp per row, whose staged query row is sqw. crow / cvrow
// are the row's `slots` candidate chunks and their approximate maxima, g / ng its gallery. Distances in the FDLNet form; ties
// resolve to the lower gallery index like torch.min / a stable sort. rerank_kernel and rerank_batched_kernel both run this
// body, so a batched or pair-table row equals the per-pair hn_match row bit for bit.
// Known limit (documented precondition of hn_match): the GEMM keeps the kTopC = 4 best chunks per row and list (a list = one
// gallery segment, or one 64-column half of it in the CTA-pair kernel). Should five or more chunks of ONE list reach the
// threshold, the fifth is not re-ranked; with 15-30 lists per row this needs five near-tied best candidates inside one list
// (|d - d2| within the 2^-9 margin). Scanning the whole segment whenever a list's fourth chunk passes the threshold was
// measured: it fires on ~5 % of the rows of the BASELINE config-4 set and makes the call 5x slower (0.88 -> 4.2 ms), so the
// exact remedy has to track the largest DROPPED chunk maximum in the GEMM epilogue instead (not done).
// Both re-rank kernels ask for 10 CTAs per SM, i.e. at most 48 registers, which this body fits without spilling. Left to its
// own choice ptxas spilled 8 bytes in some instantiations to stay within 48 or 56 registers.
constexpr int kRerankCtasPerSm = 10;
// gallery segments of the batched GEMM (hn_match_batched) and of the top-k GEMMs: bounds their candidate lists,
// [rows][segments][kTopC or kTopKC]
constexpr int kMaxBatchedSegments = 16;
template <typename T>
__device__ __forceinline__ Top2 rerank_row(const float* sqw, const T* g, long long ng, const int* crow, const float* cvrow, int slots,
                                           float margin, int lane) {
  // A chunk can hold one of the two nearest columns only if its approximate maximum reaches the second largest
  // chunk maximum minus twice the error bound of the 16-bit-operand dot product (`margin`, same scaled units).
  float thr;
  {
    float m1 = -__int_as_float(0x7f800000), m2 = m1;
    for (int c = lane; c < slots; c += 32) {
      const float v = crow[c] >= 0 ? cvrow[c] : -__int_as_float(0x7f800000);
      if (v > m1) { m2 = m1; m1 = v; } else if (v > m2) { m2 = v; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float o1 = __shfl_xor_sync(0xffffffffu, m1, o), o2 = __shfl_xor_sync(0xffffffffu, m2, o);
      const float lo = fminf(m1, o1);
      m1 = fmaxf(m1, o1);
      m2 = fmaxf(fmaxf(m2, o2), lo);
    }
    thr = m2 - margin;   // -inf when fewer than two chunks exist: everything is re-ranked
  }
  const float inf = __int_as_float(0x7f800000);
  float b1 = inf, b2 = inf;
  int j1 = 0x7fffffff, j2 = 0x7fffffff;
  // the warp walks the surviving chunks together, every lane sees the same (d, index) stream
  const float4 qv = reinterpret_cast<const float4*>(sqw)[lane];
  auto eval_chunk = [&](long long chunk) {
    const long long col0 = chunk * kChunk, left = ng - col0;   // column col0 + r exists iff r < left
    const float mine = chunk_distance(qv, g, col0, left, lane);
#pragma unroll
    for (int r = 0; r < kChunk; ++r) {
      const float d = __shfl_sync(0xffffffffu, mine, r);
      if (r >= left) continue;
      const int ci = static_cast<int>(col0) + r;   // ng < 2^31
      if (d < b1 || (d == b1 && ci < j1)) {
        b2 = b1; j2 = j1; b1 = d; j1 = ci;
      } else if (d < b2 || (d == b2 && ci < j2)) {
        b2 = d; j2 = ci;
      }
    }
  };
  for (int c = 0; c < slots; ++c) {
    const int chunk = crow[c];
    if (chunk < 0 || cvrow[c] < thr) continue;   // warp-uniform
    eval_chunk(chunk);
  }
  return {b1, b2, j1, j2};   // the same on every lane
}

// Re-rank of hn_match: query row `row` of q against g; optional outputs, indices shifted by g_offset.
// T: fp32, fp16, bf16 or e4m3 rows (ld_row4 / ldg_row4).
template <typename T>
__global__ void __launch_bounds__(128, kRerankCtasPerSm) rerank_kernel(const T* __restrict__ q, const T* __restrict__ g,
                                                     const int* __restrict__ cand, const float* __restrict__ cand_val,
                                                     float margin, long long nq, long long ng, int slots,
                                                     long long g_offset, float* __restrict__ d1, float* __restrict__ d2,
                                                     int* __restrict__ i1, int* __restrict__ i2) {
  __shared__ __align__(16) float sq[4][128];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = static_cast<int>(blockIdx.x * 4 + w);   // nq < 2^31; widened where it scales an element offset
  if (row >= nq) return;
  reinterpret_cast<float4*>(sq[w])[lane] = ld_row4(q + static_cast<long long>(row) * 128, lane);
  __syncwarp();
  const Top2 t = rerank_row(sq[w], g, ng, cand + static_cast<long long>(row) * slots, cand_val + static_cast<long long>(row) * slots,
                            slots, margin, lane);
  if (lane == 0) {
    if (d1) d1[row] = t.d1;
    if (i1) i1[row] = t.i1 == 0x7fffffff ? -1 : static_cast<int>(t.i1 + g_offset);
    if (d2) d2[row] = t.d2;
    if (i2) i2[row] = t.i2 == 0x7fffffff ? -1 : static_cast<int>(t.i2 + g_offset);
  }
}

// Batched re-rank over the flat [B * nq_pad] query rows of hn_match_batched: row -> pair b = row / nq_pad, whose gallery is
// rows [0, g_len[b]) of g + b * ng_pad * 128; indices are local to the pair. Rows past q_len[b] get the fill values
// (d = +inf, i = -1). TABLE (hn_match_pairs): pair b's rows are the ranges of the pair table over the concatenated sets instead,
// query row qs + r of q and gallery rows [gs, gs + gl) of g_all. The padded instantiation does not read its layout through the
// table accessor: that measured 1-2 % slower.
template <bool TABLE, typename T>
__global__ void __launch_bounds__(128, kRerankCtasPerSm) rerank_batched_kernel(const T* __restrict__ q, const T* __restrict__ g_all,
                                                             const int* __restrict__ cand, const float* __restrict__ cand_val,
                                                             float margin, long long B, long long nq_pad, long long ng_pad,
                                                             const int* __restrict__ q_len, const int* __restrict__ g_len, int slots,
                                                             float* __restrict__ d1, float* __restrict__ d2, int* __restrict__ i1,
                                                             int* __restrict__ i2, const int* __restrict__ pairs, long long q_rows,
                                                             long long g_rows) {
  __shared__ __align__(16) float sq[4][128];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * 4 + w;
  if (row >= B * nq_pad) return;
  const int b = static_cast<int>(row) / static_cast<int>(nq_pad);   // B * nq_pad < 2^31; element offsets below stay 64-bit
  Span qs{0, 0}, gs{0, 0};
  if constexpr (TABLE) {
    qs = table_span(pairs, b, 0, nq_pad, q_rows);
    gs = table_span(pairs, b, 1, ng_pad, g_rows);
  }
  if (row - b * nq_pad >= (TABLE ? qs.len : pair_len(q_len, b, nq_pad))) {
    if (lane == 0) {
      d1[row] = d2[row] = __int_as_float(0x7f800000);
      i1[row] = i2[row] = -1;
    }
    return;
  }
  const T* g = TABLE ? g_all + gs.start * 128 : g_all + static_cast<long long>(b) * ng_pad * 128;
  const long long ng = TABLE ? gs.len : pair_len(g_len, b, ng_pad);
  const int* crow = cand + row * slots;
  const float* cvrow = cand_val + row * slots;
  reinterpret_cast<float4*>(sq[w])[lane] = ld_row4(q + (TABLE ? qs.start + (row - b * nq_pad) : row) * 128, lane);
  __syncwarp();
  const Top2 t = rerank_row(sq[w], g, ng, crow, cvrow, slots, margin, lane);
  if (lane == 0) {
    d1[row] = t.d1;
    i1[row] = t.i1 == 0x7fffffff ? -1 : t.i1;
    d2[row] = t.d2;
    i2[row] = t.i2 == 0x7fffffff ? -1 : t.i2;
  }
}

// ------------------------------------------------------------------------------------------------------------
// k nearest neighbours (hn_match_topk, hn_match_pairs_topk), k <= kTopKMax
// ------------------------------------------------------------------------------------------------------------
// The GEMM keeps kTopKC = 8 chunks per row and list (a list = one gallery segment) and each list's dropped maximum: the
// largest approximate chunk maximum that did not make the list. The re-rank of a row then
//   - takes M_k, the k-th largest kept chunk maximum over all of the row's lists (-inf with fewer than k kept chunks), and the
//     threshold thr = M_k - kRerankMargin;
//   - evaluates every kept chunk whose maximum is >= thr, and
//   - for every list whose dropped maximum is >= thr evaluates every chunk of that list's column range instead (fallback).
// Why this is exact. Let eps = 2^-10 bound the error of the approximate (fp16- or e4m3-operand) dot product, as for the
// margins above (kF8DotBound). The k distinct columns behind the k largest kept maxima have approximate dots >= M_k, hence
// exact dots >= M_k - eps: the k-th best exact dot is at least M_k - eps, and every column of the exact top-k has an
// approximate dot >= M_k - 2 eps. A kept chunk, or the dropped part of a list, whose maximum is below M_k - 2 eps therefore
// holds none of them; whatever holds one is evaluated. The margin is twice that, 4 eps: the second factor of two covers the
// fp32 summation of the re-rank (its error is some 1e-6 of a dot product) and distances that round to the same fp32 value, so
// the columns evaluated include the top k of a brute-force fp32 evaluation sorted by (distance, index). Nothing depends on how
// many of a list's chunks come close: a list whose ninth chunk reaches the threshold is scanned whole, and with up to
// kMaxBatchedSegments lists per row a scan covers at most 1/16 of the gallery (plus one tile).
// The running top-k lives in the warp's registers: lane j < k holds the j-th best (distance, column); a candidate finds its
// place with one ballot and the entries behind it move one lane up with a shuffle.
constexpr int kTopKMax = 8;
constexpr int kRerankTopkCtasPerSm = 6;   // up to 80 registers: at 48 (kRerankCtasPerSm) or 64 the top-k re-rank spilled
static_assert(kMaxBatchedSegments * kTopKC <= 4 * 32, "rerank_topk_row holds a row's list maxima in four registers per lane");

struct TopkEntry {
  float d;
  int i;   // 0x7fffffff: fewer columns than that
};

// One query row (staged in sqw, lanes as rerank_row): its gallery g / ng, its `segments` lists crow / cvrow ([segments][kTopKC])
// and their dropped maxima drow. Returns the lane's entry of the row's top k; `scanned` tells whether a list was scanned whole.
template <typename T>
__device__ __forceinline__ TopkEntry rerank_topk_row(const float* sqw, const T* g, long long ng, const int* crow, const float* cvrow,
                                                     const float* drow, int segments, int k, float margin, int lane, bool& scanned) {
  const float inf = __int_as_float(0x7f800000);
  const int slots = segments * kTopKC;
  // slot c = lane + 32 j of the row's lists (list c / kTopKC) is held by this lane: chunk id and maximum (-inf: unused)
  int cid[4];
  float v[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = lane + 32 * j;
    cid[j] = c < slots ? crow[c] : -1;
    v[j] = cid[j] >= 0 ? cvrow[c] : -inf;
  }
  // M_k, counting equal maxima: each round takes the largest value below the previous one and how many slots hold it
  float mk = -inf, below = inf;
  int need = k;
  for (int it = 0; it < k; ++it) {
    float m = -inf;
#pragma unroll
    for (int j = 0; j < 4; ++j) m = v[j] < below ? fmaxf(m, v[j]) : m;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (m == -inf) break;   // fewer than k kept chunks: thr = -inf, every kept chunk is evaluated
    int cnt = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) cnt += v[j] == m ? 1 : 0;
    cnt = static_cast<int>(__reduce_add_sync(0xffffffffu, static_cast<unsigned>(cnt)));
    if (cnt >= need) { mk = m; break; }
    need -= cnt;
    below = m;
  }
  const float thr = mk - margin;
  // lists whose dropped maximum reaches the threshold may hide one of the k nearest columns: their whole column range
  // (seg_range of the GEMM) is evaluated instead of their kept chunks
  const float dl = lane < segments ? drow[lane] : -inf;
  const unsigned scan = __ballot_sync(0xffffffffu, dl > -inf && dl >= thr);
  scanned = scan != 0;
  unsigned take[4];   // per j, the lanes whose slot j is a kept chunk to evaluate
#pragma unroll
  for (int j = 0; j < 4; ++j)
    take[j] = __ballot_sync(0xffffffffu, cid[j] >= 0 && v[j] >= thr && !((scan >> ((lane + 32 * j) / kTopKC)) & 1u));

  TopkEntry e{inf, 0x7fffffff};
  const float4 qv = reinterpret_cast<const float4*>(sqw)[lane];
  auto eval_chunk = [&](long long chunk) {
    const long long col0 = chunk * kChunk, left = ng - col0;   // column col0 + r exists iff r < left
    const float mine = chunk_distance(qv, g, col0, left, lane);
#pragma unroll
    for (int r = 0; r < kChunk; ++r) {
      const float d = __shfl_sync(0xffffffffu, mine, r);
      if (r >= left) continue;
      const int ci = static_cast<int>(col0) + r;   // ng < 2^31
      // the entries the candidate precedes in (d, column) order: a suffix of the k lanes, starting at its place
      const unsigned behind = __ballot_sync(0xffffffffu, lane < k && (d < e.d || (d == e.d && ci < e.i)));
      if (behind) {   // warp-uniform
        const int pos = __ffs(behind) - 1;
        const float ud = __shfl_up_sync(0xffffffffu, e.d, 1);
        const int ui = __shfl_up_sync(0xffffffffu, e.i, 1);
        if (lane > pos) e = {ud, ui};
        else if (lane == pos) e = {d, ci};
      }
    }
  };
  // One walk over the work, so that eval_chunk has one call site: the kept chunks of take[0..3], then the scanned lists'
  // ranges. Every branch is warp-uniform.
  const long long tiles = (ng + kDistTile - 1) / kDistTile, chunks = (ng + kChunk - 1) / kChunk;
  int j = 0;
  unsigned lists = scan;
  long long c = 0, c1 = 0;   // the scanned list's chunks still to evaluate
  for (;;) {
    long long chunk;
    if (j < 4) {
      const unsigned t = j == 0 ? take[0] : j == 1 ? take[1] : j == 2 ? take[2] : take[3];
      if (!t) { ++j; continue; }
      const int src = __ffs(t) - 1;
      const int held = j == 0 ? cid[0] : j == 1 ? cid[1] : j == 2 ? cid[2] : cid[3];
      if (j == 0) take[0] &= t - 1; else if (j == 1) take[1] &= t - 1; else if (j == 2) take[2] &= t - 1; else take[3] &= t - 1;
      chunk = __shfl_sync(0xffffffffu, held, src);
    } else if (c < c1) {
      chunk = c++;
    } else if (lists) {
      const int l = __ffs(lists) - 1;
      lists &= lists - 1;
      c = tiles * l / segments * (kDistTile / kChunk);
      c1 = std::min(tiles * (l + 1) / segments * (kDistTile / kChunk), chunks);
      continue;
    } else {
      break;
    }
    eval_chunk(chunk);
  }
  return e;
}

// Output of one top-k row: lane j < k writes entry j; rows that scanned a list are counted when `fallback_rows` is set.
__device__ __forceinline__ void store_topk_row(const TopkEntry& e, long long row, int k, bool scanned, float* dist, int* idx,
                                               unsigned long long* fallback_rows, int lane) {
  if (lane < k) {
    dist[row * k + lane] = e.d;
    idx[row * k + lane] = e.i == 0x7fffffff ? -1 : e.i;
  }
  if (fallback_rows && scanned && lane == 0) atomicAdd(fallback_rows, 1ull);
}

// Re-rank of hn_match_topk: query row `row` of q against g, lists [nq][segments][kTopKC] and dropped maxima [nq][segments].
template <typename T>
__global__ void __launch_bounds__(128, kRerankTopkCtasPerSm) rerank_topk_kernel(const T* __restrict__ q, const T* __restrict__ g,
                                                          const int* __restrict__ cand, const float* __restrict__ cand_val,
                                                          const float* __restrict__ cand_drop, float margin, long long nq,
                                                          long long ng, int segments, int k, float* __restrict__ dist,
                                                          int* __restrict__ idx, unsigned long long* fallback_rows) {
  __shared__ __align__(16) float sq[4][128];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * 4 + w;
  if (row >= nq) return;
  reinterpret_cast<float4*>(sq[w])[lane] = ld_row4(q + row * 128, lane);
  __syncwarp();
  bool scanned = false;
  const TopkEntry e = rerank_topk_row(sq[w], g, ng, cand + row * segments * kTopKC, cand_val + row * segments * kTopKC,
                                      cand_drop + row * segments, segments, k, margin, lane, scanned);
  store_topk_row(e, row, k, scanned, dist, idx, fallback_rows, lane);
}

// Re-rank of hn_match_pairs_topk over the flat [B * nq_pad] rows: pair b = row / nq_pad matches query row qs + r of q against
// gallery rows [gs, gs + gl) of g_all (table_span, as rerank_batched_kernel); rows past the pair's length get +inf / -1.
template <typename T>
__global__ void __launch_bounds__(128, kRerankTopkCtasPerSm) rerank_topk_pairs_kernel(const T* __restrict__ q, const T* __restrict__ g_all,
                                                                const int* __restrict__ cand, const float* __restrict__ cand_val,
                                                                const float* __restrict__ cand_drop, float margin, long long B,
                                                                long long nq_pad, long long ng_pad, const int* __restrict__ pairs,
                                                                long long q_rows, long long g_rows, int segments, int k,
                                                                float* __restrict__ dist, int* __restrict__ idx,
                                                                unsigned long long* fallback_rows) {
  __shared__ __align__(16) float sq[4][128];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * 4 + w;
  if (row >= B * nq_pad) return;
  const int b = static_cast<int>(row) / static_cast<int>(nq_pad);   // B * nq_pad < 2^31
  const Span qs = table_span(pairs, b, 0, nq_pad, q_rows), gs = table_span(pairs, b, 1, ng_pad, g_rows);
  if (row - b * nq_pad >= qs.len) {
    store_topk_row(TopkEntry{__int_as_float(0x7f800000), 0x7fffffff}, row, k, false, dist, idx, nullptr, lane);
    return;
  }
  reinterpret_cast<float4*>(sq[w])[lane] = ld_row4(q + (qs.start + (row - b * nq_pad)) * 128, lane);
  __syncwarp();
  bool scanned = false;
  const TopkEntry e = rerank_topk_row(sq[w], g_all + gs.start * 128, gs.len, cand + row * segments * kTopKC,
                                      cand_val + row * segments * kTopKC, cand_drop + row * segments, segments, k, margin, lane,
                                      scanned);
  store_topk_row(e, row, k, scanned, dist, idx, fallback_rows, lane);
}

// ------------------------------------------------------------------------------------------------------------
// radius matching (hn_match_radius_*, hn_match_pairs_radius_*): every column j with d(i, j) < r, as CSR
// ------------------------------------------------------------------------------------------------------------
// The GEMM is the top-k one (kTopKC chunks per list and each list's dropped maximum); the re-rank is rerank_topk_row's
// selection with a threshold fixed by the radius instead of derived from M_k:
//   - thr = P(r) / kDotScale - kRerankMargin, with P(r) = 1 - r^2 (1 + 2^-20) / 2 (radius_threshold, on the host);
//   - every kept chunk whose maximum is >= thr is evaluated, and every list whose dropped maximum is >= thr is evaluated over its
//     whole column range instead of its kept chunks.
// Why this is exact. d = sqrtf(min(max(fl(2 - 2p), 1e-8), 4)) with p the re-rank's fp32 dot. sqrtf is correctly rounded and r is
// an fp32 value, so d < r implies sqrt(x) < r for the clamped x, hence fl(2 - 2p) <= x < r^2; fl(y) >= y (1 - 2^-24) for y > 0
// gives 2 - 2p < r^2 / (1 - 2^-24), i.e. p > P(r) (the factor 1 + 2^-20 covers 1 / (1 - 2^-24)). The exact dot is within the
// fp32 summation error (some 1e-6) of p and the approximate dot within eps = 2^-10 of the exact one (the bound of the margins
// above), so the chunk holding j has an approximate maximum >= P(r) - 2 eps; kRerankMargin is 4 eps, and rounding thr to fp32
// moves it by less than 2^-7 of the 2^16 scaled units. So a column with d < r lies in a kept chunk at or above thr, or in the
// dropped part of a list whose dropped maximum reaches thr: it is evaluated, and the result is a brute-force evaluation of every
// column with this arithmetic, whatever the ties. Each column is evaluated at most once (the chunks of a list are distinct, lists
// cover disjoint column ranges, a scanned list's kept chunks are skipped), so no entry repeats.
// Ascending columns without a sort: the lists are walked in segment order (segment ranges ascend), a scanned list over its
// range, a kept list's taken chunks in ascending id order (one __reduce_min_sync each); inside a chunk the hits are placed with
// one ballot. The count and the fill run the same selection on the same lists, so the fill writes exactly the counted entries.
// Kept apart from rerank_topk_row rather than sharing its selection: the top-k kernels keep their instructions.
template <bool FILL, typename T>
__device__ __forceinline__ int rerank_radius_row(const float* sqw, const T* g, long long ng, const int* crow, const float* cvrow,
                                                 const float* drow, int segments, float thr, float radius, int lane, bool& scanned,
                                                 long long base, long long capacity, int* col, float* dist) {
  const float inf = __int_as_float(0x7f800000);
  const int slots = segments * kTopKC;
  // slot c = lane + 32 j (list c / kTopKC) is held by this lane; bit j of tk: a kept chunk at or above the threshold
  int cid[4];
  unsigned tk = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = lane + 32 * j;
    cid[j] = c < slots ? crow[c] : -1;
    if (cid[j] >= 0 && cvrow[c] >= thr) tk |= 1u << j;
  }
  const float dl = lane < segments ? drow[lane] : -inf;
  const unsigned scan = __ballot_sync(0xffffffffu, dl > -inf && dl >= thr);
  scanned = scan != 0;

  int n = 0;   // entries of the row so far
  const float4 qv = reinterpret_cast<const float4*>(sqw)[lane];
  auto eval_chunk = [&](long long chunk) {
    const long long col0 = chunk * kChunk, left = ng - col0;   // column col0 + r exists iff r < left
    const float mine = chunk_distance(qv, g, col0, left, lane);   // lane r < kChunk: column col0 + r
    const bool hit = lane < kChunk && lane < left && mine < radius;
    const unsigned hits = __ballot_sync(0xffffffffu, hit);
    if (FILL && hit) {
      const long long pos = base + n + __popc(hits & ((1u << lane) - 1u));
      if (pos < capacity) {
        col[pos] = static_cast<int>(col0) + lane;   // ng < 2^31
        if (dist) dist[pos] = mine;
      }
    }
    n += __popc(hits);
  };
  // One walk, so that eval_chunk has one call site: list l = 0, 1, ... either as its range [c, c1) or as its taken chunks, which
  // the lanes of slots l * kTopKC ... (lanes 8 (l % 4) ... of j = l / 4) offer in `offer` and the warp takes smallest first.
  const long long tiles = (ng + kDistTile - 1) / kDistTile, chunks = (ng + kChunk - 1) / kChunk;
  constexpr int kNone = 0x7fffffff;
  int l = 0, offer = kNone;
  long long c = 0, c1 = 0;
  for (;;) {
    long long chunk;
    if (c < c1) {
      chunk = c++;
    } else {
      const int m = __reduce_min_sync(0xffffffffu, offer);
      if (m != kNone) {
        chunk = m;
        if (offer == m) offer = kNone;
      } else if (l < segments) {
        if ((scan >> l) & 1u) {
          c = tiles * l / segments * (kDistTile / kChunk);
          c1 = std::min(tiles * (l + 1) / segments * (kDistTile / kChunk), chunks);
        } else {
          const int j = l >> 2;
          const int held = j == 0 ? cid[0] : j == 1 ? cid[1] : j == 2 ? cid[2] : cid[3];
          offer = (lane >> 3) == (l & 3) && ((tk >> j) & 1u) ? held : kNone;
        }
        ++l;
        continue;
      } else {
        break;
      }
    }
    eval_chunk(chunk);
  }
  return n;
}

// Count (FILL = false) or fill of hn_match_radius_* (TABLE = false: `rows` query rows of q against ng_pad gallery rows of g_all)
// and hn_match_pairs_radius_* (TABLE: pair b = row / nq_pad, ranges from the table as rerank_topk_pairs_kernel). Lists
// [rows][segments][kTopKC], dropped maxima [rows][segments]. The count writes row i's number of entries to row_ptr[i + 1] (rows
// past q_len: 0); the fill writes row i's entries from position row_ptr[i] on, those below `capacity`.
template <bool TABLE, bool FILL, typename T>
__global__ void __launch_bounds__(128, kRerankTopkCtasPerSm) rerank_radius_kernel(
    const T* __restrict__ q, const T* __restrict__ g_all, const int* __restrict__ cand, const float* __restrict__ cand_val,
    const float* __restrict__ cand_drop, float thr, float radius, long long rows, long long nq_pad, long long ng_pad,
    const int* __restrict__ pairs, long long q_rows, long long g_rows, int segments, long long* __restrict__ row_ptr,
    long long capacity, int* __restrict__ col, float* __restrict__ dist, unsigned long long* fallback_rows) {
  __shared__ __align__(16) float sq[4][128];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * 4 + w;
  if (row >= rows) return;
  long long base = 0;
  if constexpr (FILL) {
    base = row_ptr[row];
    if (row_ptr[row + 1] == base || base >= capacity) return;   // nothing of this row to write
  } else {
    if (row == 0 && lane == 0) row_ptr[0] = 0;
  }
  const T* qrow = q + row * 128;
  const T* g = g_all;
  long long ng = ng_pad;
  if constexpr (TABLE) {
    const int b = static_cast<int>(row) / static_cast<int>(nq_pad);   // B * nq_pad < 2^31
    const Span qs = table_span(pairs, b, 0, nq_pad, q_rows), gs = table_span(pairs, b, 1, ng_pad, g_rows);
    if (row - b * nq_pad >= qs.len || gs.len == 0) {
      if (!FILL && lane == 0) row_ptr[row + 1] = 0;
      return;
    }
    qrow = q + (qs.start + (row - b * nq_pad)) * 128;
    g = g_all + gs.start * 128;
    ng = gs.len;
  }
  reinterpret_cast<float4*>(sq[w])[lane] = ld_row4(qrow, lane);
  __syncwarp();
  bool scanned = false;
  const int n = rerank_radius_row<FILL>(sq[w], g, ng, cand + row * segments * kTopKC, cand_val + row * segments * kTopKC,
                                        cand_drop + row * segments, segments, thr, radius, lane, scanned, base, capacity, col, dist);
  if (!FILL && lane == 0) {
    row_ptr[row + 1] = n;
    if (fallback_rows && scanned) atomicAdd(fallback_rows, 1ull);
  }
}

// Exclusive scan of the radius counts into row offsets, in place over x = row_ptr + 1 ([n] counts -> [n] inclusive sums): tile
// sums, an exclusive scan of the tile sums in one block, then each tile's inclusive scan plus its offset. A thread owns kScanItems
// consecutive elements of a kScanTile-element tile.
constexpr int kScanThreads = 1024, kScanItems = 8, kScanTile = kScanThreads * kScanItems;

// Inclusive scan of v over the block (kScanThreads threads); *total receives the block's sum. s: 32 words of shared memory.
__device__ __forceinline__ long long block_inclusive_scan(long long v, long long* s, long long* total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  if (lane == 31) s[w] = v;
  __syncthreads();
  if (w == 0) {
    long long x = s[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long t = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += t;
    }
    s[lane] = x;
  }
  __syncthreads();
  if (w > 0) v += s[w - 1];
  *total = s[31];
  __syncthreads();   // s is reused by the caller's next scan
  return v;
}

__global__ void __launch_bounds__(kScanThreads) scan_tile_sum_kernel(const long long* __restrict__ x, long long n,
                                                                     long long* __restrict__ tile_sum) {
  __shared__ long long s[32];
  const long long i0 = static_cast<long long>(blockIdx.x) * kScanTile + threadIdx.x * kScanItems;
  long long v = 0;
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) v += i0 + k < n ? x[i0 + k] : 0;
  long long total;
  block_inclusive_scan(v, s, &total);
  if (threadIdx.x == 0) tile_sum[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kScanThreads) scan_tile_offsets_kernel(long long* __restrict__ tile_sum, long long tiles) {
  __shared__ long long s[32];
  long long carry = 0;
  for (long long t0 = 0; t0 < tiles; t0 += kScanThreads) {
    const long long t = t0 + threadIdx.x;
    const long long v = t < tiles ? tile_sum[t] : 0;
    long long total;
    const long long incl = block_inclusive_scan(v, s, &total);
    if (t < tiles) tile_sum[t] = carry + incl - v;
    carry += total;
  }
}

__global__ void __launch_bounds__(kScanThreads) scan_tile_apply_kernel(long long* __restrict__ x, long long n,
                                                                       const long long* __restrict__ tile_off) {
  __shared__ long long s[32];
  const long long i0 = static_cast<long long>(blockIdx.x) * kScanTile + threadIdx.x * kScanItems;
  long long v[kScanItems], sum = 0;
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) {
    v[k] = i0 + k < n ? x[i0 + k] : 0;
    sum += v[k];
  }
  long long total;
  long long run = block_inclusive_scan(sum, s, &total) - sum + tile_off[blockIdx.x];
#pragma unroll
  for (int k = 0; k < kScanItems; ++k) {
    run += v[k];
    if (i0 + k < n) x[i0 + k] = run;
  }
}

// Process-wide count of top-k rows that scanned a list (hn_match_topk_fallback_*): off by default (nullptr), else a device word
// of the device that was current when it was enabled. Not a __device__ variable: that would move the constant-bank addresses
// every other kernel of this file uses.
static unsigned long long* g_topk_fallback_rows = nullptr;
static int topk_fallback_counter(unsigned long long** p) {
  *p = g_topk_fallback_rows;
  return HN_OK;
}

// Optional per-stage CUDA-event timing of hn_match (bench.py: the roofline of the matching GEMM is computed from the kernel's
// own in-run time): stage 0 = operand packing, 1 = GEMM + shortlist, 2 = exact re-rank.
struct MatchProfile {
  bool on = false;
  std::vector<cudaEvent_t> ev[3];
  size_t used[3] = {0, 0, 0};
};
static MatchProfile g_match_profile;
struct MatchTimer {
  int stage;
  cudaStream_t s;
  bool on;
  MatchTimer(int stage_, cudaStream_t s_) : stage(stage_), s(s_), on(g_match_profile.on) { if (on) record(); }
  ~MatchTimer() { if (on) record(); }
  void record() {
    auto& v = g_match_profile.ev[stage];
    size_t& u = g_match_profile.used[stage];
    if (u == v.size()) {
      cudaEvent_t e;
      if (cudaEventCreate(&e) != cudaSuccess) { on = false; return; }
      v.push_back(e);
    }
    cudaEventRecord(v[u++], s);
  }
};


// ------------------------------------------------------------------------------------------------------------
// mutual nearest neighbours from ONE GEMM (column side: claims + verification against the block maxima)
// ------------------------------------------------------------------------------------------------------------
// claim[j] = min over the queries i whose nearest gallery row is j of (distance bits << 32 | global query row): only the best
// claimant of a column can be its mutual partner. `claim` must be initialised to an "unclaimed" value: any word whose upper
// half is >= 0x7F000000 (no real distance has such bits): bytes of 0x7F, or INT64_MAX - positive as a signed integer too, so
// that an all_reduce(MIN) over int64 orders claims like the unsigned atomicMin does.
// The claim of one query row, shared by mutual_claim_kernel and mutual_claim_batched_kernel: a warp is one 32-row block of one
// problem, whose minimum d2 over its valid rows goes to rb_min_d2[rb] (lane 0, if store_min). Row i of i1 / d1 / d2 is valid iff
// it is a row of the problem; it then claims its nearest column j < ng() of `claim` as row number id.
template <typename Cols>
__device__ __forceinline__ void claim_row(const int* i1, const float* d1, const float* d2, long long i, bool valid, float* rb_min_d2,
                                          long long rb, bool store_min, unsigned long long* claim, Cols ng, unsigned int id) {
  // a warp is one 32-row block: its smallest second-nearest distance bounds every d(k, j) with j not the nearest column of k
  float m = valid ? d2[i] : __int_as_float(0x7f800000);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && store_min) rb_min_d2[rb] = m;
  if (!valid) return;
  const long long j = i1[i];
  if (j < 0 || j >= ng()) return;
  atomicMin(claim + j, (static_cast<unsigned long long>(__float_as_uint(d1[i])) << 32) | id);
}

__global__ void mutual_claim_kernel(const int* __restrict__ i1, const float* __restrict__ d1, const float* __restrict__ d2,
                                    long long nq, long long q_offset, unsigned long long* __restrict__ claim, long long ng,
                                    float* __restrict__ rb_min_d2) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  claim_row(i1, d1, d2, i, i < nq, rb_min_d2, i >> 5, i < nq, claim, [&] { return ng; }, static_cast<unsigned int>(i + q_offset));
}

// Is the claimant of column j really the nearest query of g_j (lowest row wins ties, like torch.min)? A query row k can beat
// it only if BOTH hold: (1) dot(q_k, g_j) >= dot(claimant), and then the GEMM's (32-row block, 8-column chunk) maximum of k's
// cell is at least that dot product minus the error bound of the fp16-operand product; (2) k's own second-nearest distance
// d2[k] <= d(claimant, j): j is not k's nearest column (else k is a claimant itself and lost the atomicMin), so d(k, j) is at
// least k's second-smallest distance. (2) is what makes confident matches free: a claim at distance 0.4 is never challenged
// by rows whose second-nearest gallery row is 1.1 away, whatever their cell maximum says. One warp per chunk: scan the chunk's
// block maxima and the row blocks' minimum d2 (both contiguous), evaluate the exact fp32 distances of the cells passing both
// tests, stop as soon as every claimed column is decided.
// A cell's 32 query rows are staged ONCE in shared memory with coalesced loads (row pitch 132 floats: the per-row reads below
// are bank-conflict free; per-lane global reads at a 512-byte stride cost 32 L1 wavefronts per instruction and made this
// kernel slower than a whole second GEMM) and serve every column of the chunk that needs the cell, two columns per sweep.
// The dot product is summed in the order of rerank_row (32 float4 partials, then the xor-butterfly tree), so a distance
// computed here is bit-identical to the one a second (gallery x queries) matching pass would produce.
constexpr int kVerifyWarps = 1;   // one warp per CTA: a chunk with a weakly claimed column evaluates ~20 cells one after the other (~70 us), so CTAs must be small and many (10 per SM by shared memory) for the hardware to balance them
constexpr int kVerifyPitch = 132;   // floats per staged query row
constexpr size_t kVerifySmem = static_cast<size_t>(kVerifyWarps) * (32 * kVerifyPitch * 4 + kChunk * 32 * 16);

// Verification of the claims of column chunk cb of one problem (see above; nothing to do for a chunk past ng): q / nq, g / ng
// and the claims, cell maxima (row pitch bm_pitch, n_row_blocks of them per chunk), row blocks' minimum d2 and beaten flags of
// that problem; q_offset shifts its query rows to the rows of the claims. s_q / s_g: the warp's staging tiles.
// mutual_verify_kernel and mutual_verify_batched_kernel both run this body, so a batched or pair-table flag equals the
// per-pair one bit for bit.
template <typename T>
__device__ __forceinline__ void verify_chunk(const T* q, long long nq, long long q_offset, const T* g, long long ng,
                                             const unsigned long long* claim, const float* block_max, long long bm_pitch,
                                             const float* rb_min_d2, int n_row_blocks, float margin_scaled, float inv_dot_scale, unsigned char* beaten,
                                             long long cb, float* s_q, float4* s_g, int lane) {
  if (cb * kChunk >= ng) return;
  unsigned long long cl = 0x7FFFFFFFFFFFFFFFull;   // unclaimed
  if (lane < kChunk && cb * kChunk + lane < ng) cl = claim[cb * kChunk + lane];
  float dcl[kChunk], thr[kChunk];
  unsigned int icl[kChunk];
  unsigned undecided = 0, lost = 0;
  const float ninf = -__int_as_float(0x7f800000);
#pragma unroll
  for (int c = 0; c < kChunk; ++c) {
    const unsigned long long cc = __shfl_sync(0xffffffffu, cl, c);
    dcl[c] = __uint_as_float(static_cast<unsigned int>(cc >> 32));
    icl[c] = static_cast<unsigned int>(cc & 0xffffffffu);
    thr[c] = __int_as_float(0x7f800000);
    if ((cc >> 32) < 0x7F000000ull) {
      undecided |= 1u << c;
      thr[c] = (1.0f - 0.5f * dcl[c] * dcl[c]) * inv_dot_scale - margin_scaled;
      s_g[c * 32 + lane] = ldg_row4(g + (cb * kChunk + c) * 128, lane);
    }
  }
  if (!undecided) return;
  __syncwarp();
  const float* bm_row = block_max + cb * bm_pitch;

  // distance of this lane's staged row to column c (arithmetic of rerank_row)
  auto row_distance = [&](int c) {
    float p[32];
    const float* qr = s_q + lane * kVerifyPitch;
#pragma unroll
    for (int l = 0; l < 32; ++l) {
      const float4 qv = *reinterpret_cast<const float4*>(qr + 4 * l);
      const float4 gv = s_g[c * 32 + l];
      p[l] = fmaf(qv.x, gv.x, fmaf(qv.y, gv.y, fmaf(qv.z, gv.z, qv.w * gv.w)));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int l = 0; l < o; ++l) p[l] += p[l + o];
    }
    return sqrtf(fminf(fmaxf(2.0f - 2.0f * p[0], 1e-8f), 4.0f));
  };

  auto evaluate = [&](int rb, float vb, float min_d2) {
    unsigned need = 0;
#pragma unroll
    for (int c = 0; c < kChunk; ++c)
      if (((undecided >> c) & 1u) && thr[c] <= vb && min_d2 <= dcl[c]) need |= 1u << c;
    if (!need) return;
    // stage the cell's 32 rows: one coalesced 512-byte row per iteration
    const long long k0 = static_cast<long long>(rb) * 32;
#pragma unroll
    for (int r0 = 0; r0 < 32; r0 += 8) {   // eight row loads in flight
      float4 v[8];
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        v[r] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k0 + r0 + r < nq) v[r] = ldg_row4(q + (k0 + r0 + r) * 128, lane);
      }
#pragma unroll
      for (int r = 0; r < 8; ++r) *reinterpret_cast<float4*>(s_q + (r0 + r) * kVerifyPitch + 4 * lane) = v[r];
    }
    __syncwarp();
    const long long k = k0 + lane;
    const bool valid = k < nq;
    const unsigned int gk = static_cast<unsigned int>(k + q_offset);
#pragma unroll 1
    for (int c = 0; c < kChunk; ++c) {
      if (!((need >> c) & 1u)) continue;   // warp-uniform
      const float d = row_distance(c);
      const bool beats = valid && gk != icl[c] && (d < dcl[c] || (d == dcl[c] && gk < icl[c]));
      if (__any_sync(0xffffffffu, beats)) {
        undecided &= ~(1u << c);
        lost |= 1u << c;
      }
    }
    __syncwarp();   // the staging tile is reused by the next cell
  };

  for (int base = 0; base < n_row_blocks && undecided; base += 32) {
    const int rb = base + lane;
    const float v = rb < n_row_blocks ? bm_row[rb] : ninf;
    const float md2 = rb < n_row_blocks ? rb_min_d2[rb] : __int_as_float(0x7f800000);
    bool mine = false;
#pragma unroll
    for (int c = 0; c < kChunk; ++c) mine |= ((undecided >> c) & 1u) && thr[c] <= v && md2 <= dcl[c];
    unsigned cand = __ballot_sync(0xffffffffu, mine);
    while (cand && undecided) {
      const int b = __ffs(cand) - 1;
      cand &= cand - 1;
      evaluate(base + b, __shfl_sync(0xffffffffu, v, b), __shfl_sync(0xffffffffu, md2, b));
    }
  }
  if (lane < kChunk && ((lost >> lane) & 1u)) beaten[cb * kChunk + lane] = 1;
}

template <typename T>
__global__ void __launch_bounds__(kVerifyWarps * 32) mutual_verify_kernel(const T* __restrict__ q, long long nq, long long q_offset,
                                                                         const T* __restrict__ g, long long ng,
                                                                         const unsigned long long* __restrict__ claim,
                                                                         const float* __restrict__ block_max,
                                                                         const float* __restrict__ rb_min_d2, int n_row_blocks,
                                                                         float margin_scaled, float inv_dot_scale,
                                                                         unsigned char* __restrict__ beaten) {
  extern __shared__ __align__(16) uint8_t vsm[];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* s_q = reinterpret_cast<float*>(vsm) + static_cast<size_t>(w) * 32 * kVerifyPitch;                       // [32][132]
  float4* s_g = reinterpret_cast<float4*>(vsm + static_cast<size_t>(kVerifyWarps) * 32 * kVerifyPitch * 4) + w * kChunk * 32;   // [8][32]
  const long long cb = static_cast<long long>(blockIdx.x) * kVerifyWarps + w;
  verify_chunk(q, nq, q_offset, g, ng, claim, block_max, n_row_blocks, rb_min_d2, n_row_blocks, margin_scaled, inv_dot_scale,
               beaten, cb, s_q, s_g, lane);
}

// mutual flag of query row `row` of a problem whose nearest column is j: the best claimant of column j < ng() is the row
// (number row + q_offset in the claims), and nobody beat it. Shared by mutual_final_kernel and mutual_final_batched_kernel.
template <typename Cols>
__device__ __forceinline__ bool is_mutual(long long j, Cols ng, const unsigned long long* claim, const unsigned char* beaten,
                                          long long row, long long q_offset) {
  return j >= 0 && j < ng() && static_cast<unsigned int>(claim[j] & 0xffffffffu) == static_cast<unsigned int>(row + q_offset) &&
         !beaten[j];
}

__global__ void mutual_final_kernel(const int* __restrict__ i1, long long nq, long long q_offset,
                                    const unsigned long long* __restrict__ claim, const unsigned char* __restrict__ beaten,
                                    long long ng, unsigned char* __restrict__ mutual) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= nq) return;
  mutual[i] = is_mutual(i1[i], [&] { return ng; }, claim, beaten, i, q_offset) ? 1 : 0;
}

// Batched column side of hn_match_batched. Claims, beaten flags and block maxima are per pair ([B][ng], [B][ng],
// [B][ceil(ng / 8)][ceil(nq / 32)]); query rows are local to the pair, so ties resolve to the lowest local row as in a per-pair
// call. Rows past q_len[b] are never claimants or candidates, and columns past g_len[b] are never claimed.
// TABLE: the lengths come from the pair table (see rerank_batched_kernel); everything else is per pair as above.
// Claims: one thread per (pair, 32-row block slot): a warp is one row block of one pair, padded to whole blocks.
template <bool TABLE>
__global__ void mutual_claim_batched_kernel(const int* __restrict__ i1, const float* __restrict__ d1, const float* __restrict__ d2,
                                            long long B, long long nq, long long ng, const int* __restrict__ q_len,
                                            const int* __restrict__ g_len, unsigned long long* __restrict__ claim,
                                            float* __restrict__ rb_min_d2, const int* __restrict__ pairs, long long q_rows,
                                            long long g_rows) {
  const long long nrb = (nq + 31) / 32;
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= B * nrb * 32) return;   // whole warps
  const long long b = t / (nrb * 32), r = t - b * nrb * 32;   // 64-bit: B * nrb * 32 may pass 2^31 while B * nq does not
  const long long i = b * nq + r;
  const bool valid = r < (TABLE ? table_span(pairs, b, 0, nq, q_rows).len : pair_len(q_len, b, nq));
  const auto ng_b = [&] { return TABLE ? table_span(pairs, b, 1, ng, g_rows).len : pair_len(g_len, b, ng); };
  claim_row(i1, d1, d2, i, valid, rb_min_d2, b * nrb + (r >> 5), true, claim + b * ng, ng_b, static_cast<unsigned int>(r));
}

// One warp per (pair, 8-column chunk), scanning only the pair's valid row blocks: verify_chunk on the pair's rows, with local
// query rows (q_offset = 0) and a block_max row pitch of ceil(nq_pad / 32).
template <bool TABLE, typename T>
__global__ void __launch_bounds__(kVerifyWarps * 32) mutual_verify_batched_kernel(const T* __restrict__ q_all, const T* __restrict__ g_all,
                                                                                 long long B, long long nq_pad, long long ng_pad,
                                                                                 const int* __restrict__ q_len, const int* __restrict__ g_len,
                                                                                 const unsigned long long* __restrict__ claim_all,
                                                                                 const float* __restrict__ block_max_all,
                                                                                 const float* __restrict__ rb_min_d2_all, float margin_scaled,
                                                                                 float inv_dot_scale, unsigned char* __restrict__ beaten_all,
                                                                                 const int* __restrict__ pairs, long long q_rows, long long g_rows) {
  extern __shared__ __align__(16) uint8_t vsm[];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* s_q = reinterpret_cast<float*>(vsm) + static_cast<size_t>(w) * 32 * kVerifyPitch;                       // [32][132]
  float4* s_g = reinterpret_cast<float4*>(vsm + static_cast<size_t>(kVerifyWarps) * 32 * kVerifyPitch * 4) + w * kChunk * 32;   // [8][32]
  const long long chunks = (ng_pad + kChunk - 1) / kChunk, bm_pitch = (nq_pad + 31) / 32;
  const long long item = static_cast<long long>(blockIdx.x) * kVerifyWarps + w;
  const long long pair = static_cast<int>(item) / static_cast<int>(chunks), cb = item - pair * chunks;   // B * chunks <= B * ng_pad < 2^31
  if (pair >= B) return;
  Span qs{0, 0}, gs{0, 0};
  if constexpr (TABLE) {
    qs = table_span(pairs, pair, 0, nq_pad, q_rows);
    gs = table_span(pairs, pair, 1, ng_pad, g_rows);
  }
  const long long nq = TABLE ? qs.len : pair_len(q_len, pair, nq_pad), ng = TABLE ? gs.len : pair_len(g_len, pair, ng_pad);
  const int n_row_blocks = static_cast<int>((nq + 31) / 32);
  const T* q = TABLE ? q_all + qs.start * 128 : q_all + pair * nq_pad * 128;
  const T* g = TABLE ? g_all + gs.start * 128 : g_all + pair * ng_pad * 128;
  const unsigned long long* claim = claim_all + pair * ng_pad;
  const float* block_max = block_max_all + pair * chunks * bm_pitch;
  const float* rb_min_d2 = rb_min_d2_all + pair * bm_pitch;
  unsigned char* beaten = beaten_all + pair * ng_pad;
  verify_chunk(q, nq, 0, g, ng, claim, block_max, bm_pitch, rb_min_d2, n_row_blocks, margin_scaled, inv_dot_scale,
               beaten, cb, s_q, s_g, lane);
}


template <bool TABLE>
__global__ void mutual_final_batched_kernel(const int* __restrict__ i1, long long B, long long nq, long long ng,
                                            const int* __restrict__ q_len, const int* __restrict__ g_len,
                                            const unsigned long long* __restrict__ claim, const unsigned char* __restrict__ beaten,
                                            unsigned char* __restrict__ mutual, const int* __restrict__ pairs, long long q_rows,
                                            long long g_rows) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= B * nq) return;
  const long long b = static_cast<int>(i) / static_cast<int>(nq), r = i - b * nq;
  const bool valid = r < (TABLE ? table_span(pairs, b, 0, nq, q_rows).len : pair_len(q_len, b, nq));
  const auto ng_b = [&] { return TABLE ? table_span(pairs, b, 1, ng, g_rows).len : pair_len(g_len, b, ng); };
  mutual[i] = valid && is_mutual(i1[i], ng_b, claim + b * ng, beaten + b * ng, r, 0) ? 1 : 0;
}

// Which matching GEMM runs: -1 = by problem size, 0 = single-CTA kernel, 1 = CTA-pair kernel. The initial value comes from
// HN_MATCH_PAIR, read ONCE when first needed; tests switch it through hn_match_force_kernel instead of the environment.
static int& match_kernel_mode() {
  static int mode = [] { const char* pe = getenv("HN_MATCH_PAIR"); return pe ? atoi(pe) : -1; }();
  return mode;
}

static inline long long batched_max_segments(long long Ng) {
  return std::max<long long>(1, std::min<long long>(kMaxBatchedSegments, (Ng + kDistTile - 1) / kDistTile));
}

// Tensor map over packed operand rows of K elements: fp16 (K = 128 or 384) or, with f8, e4m3 (K = 128). 2-D [rows][K], or with
// B > 0 3-D [B][rows][K] (hn_match_batched: a box never reaches into the next pair, TMA zero-fills past `rows`). A box is one
// 128-byte K block, i.e. one 128B-swizzle atom per row, of box_rows rows.
static int make_operand_map(CUtensorMap* tm, const void* base, bool f8, int K, long long rows, long long B, int box_rows) {
  const uint64_t esz = f8 ? 1 : 2;
  const uint64_t dims[3] = {static_cast<uint64_t>(K), static_cast<uint64_t>(rows), static_cast<uint64_t>(B)};
  const uint64_t str[2] = {K * esz, static_cast<uint64_t>(rows) * K * esz};
  const uint32_t box[3] = {static_cast<uint32_t>(128 / esz), static_cast<uint32_t>(box_rows), 1};
  const int rank = B > 0 ? 3 : 2;
  return f8 ? make_tmap_8bit(tm, base, rank, dims, str, box, 128) : make_tmap_16bit(tm, base, rank, dims, str, box, 128);
}

// The shortlist GEMM's part of DistParams (hn_match, hn_match_batched, hn_match_pairs): candidate lists, optional cell maxima
// (mutual NN), Na query rows against Nb gallery rows (per-pair maxima in a batched call) and f8 = e4m3 operands. The tensor maps,
// the segment count and the batch fields are the caller's.
static DistParams shortlist_params(bool f8, long long Na, long long Nb, int* cand, float* cand_val, float* block_max) {
  DistParams dp;
  memset(&dp, 0, sizeof(dp));
  dp.side[0].cand = cand;
  dp.side[0].cand_val = cand_val;
  dp.side[0].block_max = block_max;
  dp.side[0].n_row_blocks = static_cast<int>((Na + 31) / 32);
  dp.side[0].Na = Na;
  dp.side[0].Nb = Nb;
  dp.k_blocks = f8 ? 1 : 2;
  dp.form = HN_FORM_FDL;
  dp.dot_scale = kDotScale;
  return dp;
}

template <int MB, int EPI, bool F8 = false, int TOPC = kTopC>
static int launch_dist(const DistParams& p, int grid_x, int grid_y, cudaStream_t s) {
  auto kern = dist_kernel<MB, EPI, F8, TOPC>;
  const size_t smem = dist_smem_bytes<MB>(p.k_blocks);
  // the size depends on k_blocks (MB = 1: up to 6 for the 3-way split, MB = 2: always 2): raise the limit once per device
  static DeviceOnce attr_once;
  if (attr_once.first_time())
    HN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(dist_smem_bytes<MB>(MB == 1 ? 6 : 2))));
  kern<<<dim3(grid_x, grid_y), 64 + 128 * MB * dist_col_split<EPI>(), smem, s>>>(p);
  HN_CUDA(cudaGetLastError());
  count_launch();
  return HN_OK;
}

struct ExactWs {
  uint16_t *a16, *p16;
  float *na, *np, *pos;
  unsigned long long *row_pack, *col_pack;
  size_t bytes;
};

static ExactWs carve_exact(void* ws, long long Na, long long Np) {
  ExactWs w;
  char* b = static_cast<char*>(ws);
  size_t off = 0;
  auto take = [&](size_t n) { char* r = b ? b + off : nullptr; off += align256(n); return r; };
  w.a16 = reinterpret_cast<uint16_t*>(take(static_cast<size_t>(Na) * 384 * 2));
  w.p16 = reinterpret_cast<uint16_t*>(take(static_cast<size_t>(Np) * 384 * 2));
  w.na = reinterpret_cast<float*>(take(static_cast<size_t>(Na) * 4));
  w.np = reinterpret_cast<float*>(take(static_cast<size_t>(Np) * 4));
  w.pos = reinterpret_cast<float*>(take(static_cast<size_t>(std::max(Na, Np)) * 4));
  w.row_pack = reinterpret_cast<unsigned long long*>(take(static_cast<size_t>(Na) * 8));
  w.col_pack = reinterpret_cast<unsigned long long*>(take(static_cast<size_t>(Np) * 8));
  w.bytes = off;
  return w;
}

// Workspace of a matching call: carve_match (hn_match, hn_match_mutual) or carve_batched (hn_match_batched, hn_match_pairs).
struct MatchWs {
  void *q16, *g16;           // packed operand slots of 256 bytes per row (fp16; e4m3 operands use the first half of each)
  int* cand;
  float* cand_val;
  float* cand_drop;          // top-k only: the lists' dropped maxima
  float* block_max;          // mutual only
  unsigned long long* claim;
  unsigned char* beaten;
  float* rb_min_d2;
  size_t bytes;
};

// hn_match: packed operands and candidate lists [Nq][<= 16 segments][2 lists in the CTA-pair kernel][kTopC]. One workspace
// serves this layout and carve_exact (hn_dist_workspace_bytes), plus 256 bytes. with_mutual (hn_match_mutual): the column side's
// cell maxima, claims, beaten flags and row blocks' minimum d2 follow that size, plus 256 bytes. width = kTopKC (hn_match_topk):
// lists [Nq][<= 16 segments][kTopKC] (single-CTA kernel only) and their dropped maxima [Nq][<= 16 segments] instead.
static MatchWs carve_match(void* ws, long long Nq, long long Ng, bool with_mutual, int width = kTopC) {
  MatchWs w{};
  char* b = static_cast<char*>(ws);
  size_t off = 0;
  auto take = [&](size_t n) { char* r = b ? b + off : nullptr; off += align256(n); return r; };
  const size_t lists = static_cast<size_t>(Nq) * (width == kTopC ? 2 * kMaxBatchedSegments : kMaxBatchedSegments);
  w.q16 = take(static_cast<size_t>(Nq) * 128 * 2);
  w.g16 = take(static_cast<size_t>(Ng) * 128 * 2);
  w.cand = reinterpret_cast<int*>(take(lists * width * 4));
  w.cand_val = reinterpret_cast<float*>(take(lists * width * 4));
  if (width == kTopKC) w.cand_drop = reinterpret_cast<float*>(take(lists * 4));
  off = std::max(off, carve_exact(nullptr, Nq, Ng).bytes) + 256;
  if (with_mutual) {
    w.block_max = reinterpret_cast<float*>(take(static_cast<size_t>(hn_block_max_elems(Nq, Ng)) * 4));
    w.claim = reinterpret_cast<unsigned long long*>(take(static_cast<size_t>(Ng) * 8));
    w.beaten = reinterpret_cast<unsigned char*>(take(static_cast<size_t>(Ng)));
    w.rb_min_d2 = reinterpret_cast<float*>(take(static_cast<size_t>((Nq + 31) / 32) * 4));
    off += 256;
  }
  w.bytes = off;
  return w;
}

// Number of gallery segments a block of query rows is split into: work items = row blocks x segments are dealt round robin to
// `workers` persistent CTAs (or CTA pairs), so the count is chosen for the best fill of the last round (64k x 64k on 74 CTA
// pairs: 2 segments = 256 items = 3.46 rounds, i.e. 14 % of the machine idles in the last one; 15 segments = 25.9 rounds).
// Fewer segments win ties (every segment adds a shortlist per row for the re-rank to scan). A problem with fewer items than
// workers (the loss at N = 1024) simply takes the most items it can get: there the fill grows with every extra segment.
static int pick_segments(long long rows, int rows_per_block, long long cols, int workers, int max_seg) {
  const long long m_blocks = (rows + rows_per_block - 1) / rows_per_block;
  const long long n_tiles = (cols + kDistTile - 1) / kDistTile;
  const long long cap = std::max<long long>(1, std::min<long long>(max_seg, n_tiles));   // small problems: as many items as tiles allow
  int best = 1;
  double best_eff = -1.0;
  for (long long sgm = 1; sgm <= cap; ++sgm) {
    const long long items = m_blocks * sgm;
    const long long rounds = (items + workers - 1) / workers;
    const double eff = static_cast<double>(items) / static_cast<double>(rounds * workers);
    if (eff > best_eff + 0.02) { best_eff = eff; best = static_cast<int>(sgm); }
  }
  return best;
}

// desc_dtype of the matching entry points -> the element type of the row-reading kernels: f(T{}) with T = float, __half,
// __nv_bfloat16 or __nv_fp8_e4m3. check_rows has rejected every other value before.
template <typename F>
static int with_rows(int desc_dtype, F&& f) {
  if (desc_dtype == HN_F16) return f(__half{});
  if (desc_dtype == HN_BF16) return f(__nv_bfloat16{});
  if (desc_dtype == HN_F8E4M3) return f(__nv_fp8_e4m3{});
  return f(float{});
}
// Rows of type T are matched on e4m3 operands by the fp8 GEMM (e4m3 rows) or on fp16 operands (every other row type).
template <typename T>
constexpr bool kF8Rows = std::is_same<T, __nv_fp8_e4m3>::value;

// Descriptor rows of a matching call: fp32, fp16, bf16 or e4m3 (the same for both sides); 16-bit rows are read 8 bytes per
// lane, e4m3 rows 4 bytes.
static int check_rows(const char* fn, int desc_dtype, const void* a, const void* b) {
  HN_REQUIRE(desc_dtype == HN_F32 || desc_dtype == HN_F16 || desc_dtype == HN_BF16 || desc_dtype == HN_F8E4M3,
             "%s: desc_dtype must be HN_F32, HN_F16 or HN_BF16, or HN_F8E4M3 (got %d)", fn, desc_dtype);
  const uintptr_t bits = reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b);
  HN_REQUIRE(desc_dtype != HN_F16 && desc_dtype != HN_BF16 || (bits & 7) == 0, "%s: 16-bit descriptor rows must be 8-byte aligned", fn);
  HN_REQUIRE(desc_dtype != HN_F8E4M3 || (bits & 3) == 0, "%s: e4m3 descriptor rows must be 4-byte aligned", fn);
  return HN_OK;
}

// n rows of x -> their packed operand rows (fp16 [n,128], or e4m3 [n,128] for e4m3 rows). order: see pack_desc_kernel.
template <typename T>
static void launch_pack(const T* x, long long n, void* out, int order, cudaStream_t s) {
  const int threads = 256;
  const unsigned blocks = static_cast<unsigned>((n * 32 + threads - 1) / threads);
  if constexpr (kF8Rows<T>) pack_desc_f8_kernel<<<blocks, threads, 0, s>>>(x, n, static_cast<uint32_t*>(out));
  else pack_desc_kernel<<<blocks, threads, 0, s>>>(x, n, static_cast<uint16_t*>(out), 0, order, nullptr);
}

// Shared body of hn_dist_min / hn_loss_hardnet. Leaves packed minima and pos in the workspace.
static int run_exact(const float* a, const float* p, long long Na, long long Np, int form, int flags, ExactWs& w,
                     cudaStream_t s, const float* a_xy = nullptr, const float* p_xy = nullptr, float nei_c = 0.f) {
  int sm = 0;
  HN_TRY(device_sm_count(&sm));
  const int threads = 256;
  pack_desc_kernel<<<static_cast<unsigned>((Na * 32 + threads - 1) / threads), threads, 0, s>>>(a, Na, w.a16, 1, 0, w.na);
  pack_desc_kernel<<<static_cast<unsigned>((Np * 32 + threads - 1) / threads), threads, 0, s>>>(p, Np, w.p16, 1, 1, w.np);
  HN_CUDA(cudaGetLastError());
  count_launch(2);
  HN_CUDA(cudaMemsetAsync(w.row_pack, 0xff, static_cast<size_t>(Na) * 8, s));
  const bool swap = (flags & HN_FLAG_SWAP) != 0;
  if (swap) HN_CUDA(cudaMemsetAsync(w.col_pack, 0xff, static_cast<size_t>(Np) * 8, s));
  DistParams dp;
  memset(&dp, 0, sizeof(dp));
  HN_TRY(make_operand_map(&dp.side[0].tmA, w.a16, false, 384, Na, 0, kDistTile));
  HN_TRY(make_operand_map(&dp.side[0].tmB, w.p16, false, 384, Np, 0, kDistTile));
  dp.side[0].norm_a = w.na;
  dp.side[0].norm_b = w.np;
  dp.side[0].row_pack = w.row_pack;
  dp.side[0].pos = w.pos;
  dp.side[0].Na = Na;
  dp.side[0].Nb = Np;
  // transposed problem: rows = positives, columns = anchors (same packed operands, roles exchanged)
  dp.side[1].tmA = dp.side[0].tmB;
  dp.side[1].tmB = dp.side[0].tmA;
  dp.side[1].norm_a = w.np;
  dp.side[1].norm_b = w.na;
  dp.side[1].row_pack = w.col_pack;
  dp.side[1].pos = nullptr;
  dp.side[1].Na = Np;
  dp.side[1].Nb = Na;
  dp.k_blocks = 6;
  dp.form = form;
  dp.loss_mask = (flags & HN_FLAG_LOSS_MASK) ? 1 : 0;
  dp.nei_mask = (flags & HN_FLAG_NEI_MASK) ? 1 : 0;
  dp.nei_c = nei_c;
  for (int sd = 0; sd < 2; ++sd) {   // the mask is symmetric in (row, column): both directions index the same two arrays
    dp.side[sd].xy_a_rows = dp.side[sd].xy_a_cols = reinterpret_cast<const float2*>(a_xy);
    dp.side[sd].xy_p_rows = dp.side[sd].xy_p_cols = reinterpret_cast<const float2*>(p_xy);
  }
  dp.dot_scale = kDotScale;
  const long long rows = swap ? std::max(Na, Np) : Na;
  const long long cols = swap ? std::min(Na, Np) : Np;
  dp.segments = pick_segments(rows, kDistTile, cols, sm, 16);
  const long long items = ((rows + kDistTile - 1) / kDistTile) * dp.segments;
  const int grid_x = static_cast<int>(std::min<long long>(items, sm));
  if (dp.nei_mask) HN_TRY((launch_dist<1, EPI_EXACT_NEI>(dp, grid_x, swap ? 2 : 1, s)));
  else HN_TRY((launch_dist<1, EPI_EXACT>(dp, grid_x, swap ? 2 : 1, s)));
  return HN_OK;
}

}  // namespace hn

using namespace hn;

extern "C" long long hn_dist_workspace_bytes(long long Na, long long Np, int split) {
  if (Na < 0 || Np < 0) return 0;
  (void)split;
  return static_cast<long long>(carve_match(nullptr, Na, Np, false).bytes);
}

extern "C" int hn_dist_min_ex(const float* a, const float* p, long long Na, long long Np, int form, int flags, const float* a_xy,
                              const float* p_xy, float nei_c, float* pos, float* row_min, int32_t* row_arg, float* col_min,
                              int32_t* col_arg, void* workspace, long long workspace_bytes, void* stream) {
  HN_REQUIRE(a && p && workspace, "hn_dist_min: NULL argument");
  HN_REQUIRE(Na >= 1 && Np >= 1, "hn_dist_min: empty input (Na=%lld, Np=%lld)", Na, Np);
  HN_REQUIRE(Na < (1LL << 31) && Np < (1LL << 31), "hn_dist_min: more than 2^31 rows");
  HN_REQUIRE(form == HN_FORM_HARDNET || form == HN_FORM_FDL, "hn_dist_min: unknown distance form %d", form);
  HN_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "hn_dist_min: workspace must be 256-byte aligned");
  HN_REQUIRE(workspace_bytes >= hn_dist_workspace_bytes(Na, Np, 1), "hn_dist_min: workspace too small");
  if ((col_min || col_arg) && !(flags & HN_FLAG_SWAP)) {
    set_error("hn_dist_min: column outputs need HN_FLAG_SWAP");
    return HN_ERR_INVALID;
  }
  if (flags & HN_FLAG_NEI_MASK) {
    HN_REQUIRE(a_xy && p_xy && Na == Np, "hn_dist_min: the neighbour mask needs both keypoint arrays and a square problem");
    HN_REQUIRE(!(flags & HN_FLAG_LOSS_MASK), "hn_dist_min: HN_FLAG_LOSS_MASK and HN_FLAG_NEI_MASK are different losses");
    HN_REQUIRE((reinterpret_cast<uintptr_t>(a_xy) & 7) == 0 && (reinterpret_cast<uintptr_t>(p_xy) & 7) == 0,
               "hn_dist_min: keypoint arrays must be 8-byte aligned");
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  ExactWs w = carve_exact(workspace, Na, Np);
  HN_TRY(run_exact(a, p, Na, Np, form, flags, w, s, a_xy, p_xy, nei_c));
  const int threads = 256;
  if (row_min || row_arg)
    unpack_min_kernel<<<static_cast<unsigned>((Na + threads - 1) / threads), threads, 0, s>>>(w.row_pack, Na, row_min, row_arg);
  if (col_min || col_arg)
    unpack_min_kernel<<<static_cast<unsigned>((Np + threads - 1) / threads), threads, 0, s>>>(w.col_pack, Np, col_min, col_arg);
  if (pos && (flags & (HN_FLAG_LOSS_MASK | HN_FLAG_NEI_MASK)))
    HN_CUDA(cudaMemcpyAsync(pos, w.pos, static_cast<size_t>(std::min(Na, Np)) * 4, cudaMemcpyDeviceToDevice, s));
  HN_CUDA(cudaGetLastError());
  return HN_OK;
}

extern "C" int hn_dist_min(const float* a, const float* p, long long Na, long long Np, int form, int flags, float* pos,
                           float* row_min, int32_t* row_arg, float* col_min, int32_t* col_arg, void* workspace,
                           long long workspace_bytes, void* stream) {
  return hn_dist_min_ex(a, p, Na, Np, form, flags, nullptr, nullptr, 0.f, pos, row_min, row_arg, col_min, col_arg, workspace,
                        workspace_bytes, stream);
}

extern "C" int hn_loss_hardnet(const float* anchor, const float* positive, long long N, float margin, int anchor_swap,
                               float* loss_out, void* workspace, long long workspace_bytes, void* stream) {
  HN_REQUIRE(anchor && positive && loss_out && workspace, "hn_loss_hardnet: NULL argument");
  HN_REQUIRE(N >= 1 && N < (1LL << 31), "hn_loss_hardnet: N out of range (%lld)", N);
  HN_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "hn_loss_hardnet: workspace must be 256-byte aligned");
  HN_REQUIRE(workspace_bytes >= hn_dist_workspace_bytes(N, N, 1), "hn_loss_hardnet: workspace too small");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  ExactWs w = carve_exact(workspace, N, N);
  HN_TRY(run_exact(anchor, positive, N, N, HN_FORM_HARDNET, HN_FLAG_LOSS_MASK | (anchor_swap ? HN_FLAG_SWAP : 0), w, s));
  loss_finalize_kernel<<<1, 1024, 0, s>>>(w.pos, w.row_pack, anchor_swap ? w.col_pack : nullptr, N, margin, loss_out);
  HN_CUDA(cudaGetLastError());
  count_launch();
  return HN_OK;
}

// hn_pack_descriptors / hn_pack_descriptors_typed; fn names the entry point in error messages.
static int pack_entry(const char* fn, const void* x, int desc_dtype, long long n, void* out16, void* stream) {
  HN_REQUIRE(x && out16, "%s: NULL argument", fn);
  HN_TRY(check_rows(fn, desc_dtype, x, x));
  HN_REQUIRE(n >= 1 && n < (1LL << 31), "%s: n out of range (%lld)", fn, n);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return with_rows(desc_dtype, [&](auto t) -> int {
    using T = decltype(t);
    launch_pack(static_cast<const T*>(x), n, out16, 0, s);
    HN_CUDA(cudaGetLastError());
    count_launch();
    return HN_OK;
  });
}

extern "C" int hn_pack_descriptors(const float* x, long long n, void* out16, void* stream) {
  return pack_entry("hn_pack_descriptors", x, HN_F32, n, out16, stream);
}

extern "C" int hn_pack_descriptors_typed(const void* x, int desc_dtype, long long n, void* out16, void* stream) {
  return pack_entry("hn_pack_descriptors_typed", x, desc_dtype, n, out16, stream);
}

extern "C" int hn_pack_descriptors_multicast(const float* x, long long n, void* mc16, void* mc32, void* stream) {
  HN_REQUIRE(x && (mc16 || mc32), "hn_pack_descriptors_multicast: NULL argument (either destination may be NULL, not both)");
  HN_REQUIRE(n >= 1 && n < (1LL << 31), "hn_pack_descriptors_multicast: n out of range (%lld)", n);
  HN_REQUIRE((reinterpret_cast<uintptr_t>(mc16) & 15) == 0 && (reinterpret_cast<uintptr_t>(mc32) & 15) == 0,
             "hn_pack_descriptors_multicast: multicast addresses must be 16-byte aligned");
  const int threads = 256;
  pack_desc_multicast_kernel<<<static_cast<unsigned>((n * 16 + threads - 1) / threads), threads, 0, static_cast<cudaStream_t>(stream)>>>(
      x, n, static_cast<uint16_t*>(mc16), static_cast<float*>(mc32));
  HN_CUDA(cudaGetLastError());
  count_launch();
  return HN_OK;
}

// Operand packing of a single-problem call (stage 0): the packed rows the caller gave (q16_in / g16_in), else those of q / g
// packed into w.
template <typename T>
static int pack_operands(const T* q, const T* g, const void* q16_in, const void* g16_in, long long Nq, long long Ng, const MatchWs& w,
                         cudaStream_t s) {
  MatchTimer timer(0, s);
  if (!q16_in) launch_pack(q, Nq, w.q16, 0, s);
  if (!g16_in) launch_pack(g, Ng, w.g16, 1, s);
  HN_CUDA(cudaGetLastError());
  count_launch((q16_in ? 0 : 1) + (g16_in ? 0 : 1));
  return HN_OK;
}

// The launch sequence of hn_match_ex / hn_match_typed on validated arguments.
template <typename T>
static int run_match(const T* q, const T* g, const void* q16_in, const void* g16_in, long long Nq, long long Ng, long long g_offset,
                     float* d1, float* d2, int32_t* i1, int32_t* i2, float* block_max, const MatchWs& w, void* g_ready_event,
                     cudaStream_t s) {
  int sm = 0;
  HN_TRY(device_sm_count(&sm));
  constexpr bool F8 = kF8Rows<T>;
  const void* q16 = q16_in ? q16_in : w.q16;
  const void* g16 = g16_in ? g16_in : w.g16;
  HN_TRY(pack_operands(q, g, q16_in, g16_in, Nq, Ng, w, s));
  DistParams dp = shortlist_params(F8, Nq, Ng, w.cand, w.cand_val, block_max);
  // CTA pairs (tc_dist_pair.cuh) once the problem is large enough to fill the machine with 512-row query blocks
  const int pair_mode = match_kernel_mode();
  const bool use_pair = pair_mode >= 0 ? pair_mode != 0 : (Nq >= 8192 && Ng >= 1024);
  HN_TRY(make_operand_map(&dp.side[0].tmA, q16, F8, 128, Nq, 0, kDistTile));
  HN_TRY(make_operand_map(&dp.side[0].tmB, g16, F8, 128, Ng, 0, use_pair ? 64 : kDistTile));
  {
    MatchTimer timer(1, s);
    if (use_pair) {
      const int pairs = std::max(sm / 2, 1);
      dp.segments = pick_segments(Nq, 4 * kDistTile, Ng, pairs, 16);
      const long long items = ((Nq + 4 * kDistTile - 1) / (4 * kDistTile)) * dp.segments;
      static DeviceOnce attr_once;
      if (attr_once.first_time()) {
        HN_CUDA(cudaFuncSetAttribute(match_pair_kernel<F8>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(mp_smem_bytes<F8>())));
      }
      match_pair_kernel<F8><<<2 * static_cast<int>(std::min<long long>(items, pairs)), kMpThreads, mp_smem_bytes<F8>(), s>>>(dp);
      HN_CUDA(cudaGetLastError());
      count_launch();
    } else {
      dp.segments = pick_segments(Nq, 2 * kDistTile, Ng, sm, 16);
      const long long items = ((Nq + 2 * kDistTile - 1) / (2 * kDistTile)) * dp.segments;
      HN_TRY((launch_dist<2, EPI_SHORTLIST, F8>(dp, static_cast<int>(std::min<long long>(items, sm)), 1, s)));
    }
  }
  // The re-rank reads the gallery rows of the shortlisted columns; a caller that gathered the packed gallery first (half the
  // bytes of fp32 rows) passes the event that marks the rows' arrival, so that transfer hides behind the GEMM.
  if (g_ready_event) HN_CUDA(cudaStreamWaitEvent(s, static_cast<cudaEvent_t>(g_ready_event), 0));
  {
    MatchTimer timer(2, s);
    // the CTA-pair kernel keeps two top-kTopC lists per row and segment (one per 64-column half of its tiles)
    rerank_kernel<<<static_cast<unsigned>((Nq + 3) / 4), 128, 0, s>>>(q, g, w.cand, w.cand_val, kRerankMargin, Nq, Ng,
                                                                     dp.segments * kTopC * (use_pair ? 2 : 1), g_offset, d1, d2, i1, i2);
    HN_CUDA(cudaGetLastError());
    count_launch();
  }
  return HN_OK;
}

// hn_match / hn_match_ex / hn_match_typed; fn names the entry point in error messages.
// Argument checks of a single-problem matching call (hn_match_typed, hn_match_topk_typed) up to the workspace size.
static int check_match(const char* fn, int desc_dtype, const void* q, const void* g, long long Nq, long long Ng, long long g_offset,
                       const void* workspace) {
  HN_TRY(check_rows(fn, desc_dtype, q, g));
  HN_REQUIRE(Nq >= 1 && Ng >= 1, "%s: empty input (Nq=%lld, Ng=%lld)", fn, Nq, Ng);
  // a negative offset would make indices that collide with the -1 "no neighbour" fill
  HN_REQUIRE(g_offset >= 0, "%s: g_offset must be >= 0 (got %lld)", fn, g_offset);
  HN_REQUIRE(Nq < (1LL << 31) && Ng + g_offset < (1LL << 31), "%s: more than 2^31 rows", fn);
  HN_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "%s: workspace must be 256-byte aligned", fn);
  return HN_OK;
}

static int match_entry(const char* fn, const void* q, const void* g, int desc_dtype, const void* q16_in, const void* g16_in,
                       long long Nq, long long Ng, long long g_offset, float* d1, float* d2, int32_t* i1, int32_t* i2,
                       float* block_max, void* workspace, long long workspace_bytes, void* g_ready_event, void* stream) {
  HN_REQUIRE(q && g && workspace, "%s: NULL argument", fn);
  HN_TRY(check_match(fn, desc_dtype, q, g, Nq, Ng, g_offset, workspace));
  HN_REQUIRE(workspace_bytes >= hn_dist_workspace_bytes(Nq, Ng, 0), "%s: workspace too small", fn);
  HN_REQUIRE((reinterpret_cast<uintptr_t>(q16_in) & 15) == 0 && (reinterpret_cast<uintptr_t>(g16_in) & 15) == 0,
             "%s: packed operands must be 16-byte aligned", fn);
  return with_rows(desc_dtype, [&](auto t) -> int {
    using T = decltype(t);
    return run_match(static_cast<const T*>(q), static_cast<const T*>(g), q16_in, g16_in, Nq, Ng, g_offset, d1, d2, i1, i2, block_max,
                     carve_match(workspace, Nq, Ng, false), g_ready_event, static_cast<cudaStream_t>(stream));
  });
}

extern "C" int hn_match_ex(const float* q, const float* g, const void* q16_in, const void* g16_in, long long Nq, long long Ng,
                           long long g_offset, float* d1, float* d2, int32_t* i1, int32_t* i2, float* block_max, void* workspace,
                           long long workspace_bytes, void* g_ready_event, void* stream) {
  return match_entry("hn_match", q, g, HN_F32, q16_in, g16_in, Nq, Ng, g_offset, d1, d2, i1, i2, block_max, workspace, workspace_bytes,
                     g_ready_event, stream);
}

extern "C" int hn_match_typed(const void* q, const void* g, int desc_dtype, const void* q16, const void* g16, long long Nq, long long Ng,
                              long long g_offset, float* d1, float* d2, int32_t* i1, int32_t* i2, float* block_max, void* workspace,
                              long long workspace_bytes, void* g_ready_event, void* stream) {
  return match_entry("hn_match_typed", q, g, desc_dtype, q16, g16, Nq, Ng, g_offset, d1, d2, i1, i2, block_max, workspace,
                     workspace_bytes, g_ready_event, stream);
}

extern "C" int hn_match(const float* q, const float* g, long long Nq, long long Ng, long long g_offset, float* d1,
                        float* d2, int32_t* i1, int32_t* i2, void* workspace, long long workspace_bytes, void* stream) {
  return hn_match_ex(q, g, nullptr, nullptr, Nq, Ng, g_offset, d1, d2, i1, i2, nullptr, workspace, workspace_bytes, nullptr, stream);
}

extern "C" long long hn_block_max_elems(long long Nq, long long Ng) {
  if (Nq < 0 || Ng < 0) return 0;
  return ((Ng + kChunk - 1) / kChunk) * ((Nq + 31) / 32);
}

extern "C" int hn_mutual_claims(const int32_t* i1, const float* d1, const float* d2, long long Nq, long long q_offset,
                                unsigned long long* claim, long long Ng, float* rb_min_d2, void* stream) {
  HN_REQUIRE(i1 && d1 && d2 && claim && rb_min_d2, "hn_mutual_claims: NULL argument");
  // claims hold the global row as an unsigned 32-bit id: a negative offset would wrap to huge ids
  HN_REQUIRE(q_offset >= 0, "hn_mutual_claims: q_offset must be >= 0 (got %lld)", q_offset);
  HN_REQUIRE(Nq >= 1 && Ng >= 1 && Nq + q_offset < (1LL << 32), "hn_mutual_claims: size out of range");
  mutual_claim_kernel<<<static_cast<unsigned>((Nq + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(i1, d1, d2, Nq, q_offset, claim, Ng, rb_min_d2);
  HN_CUDA(cudaGetLastError());
  count_launch();
  return HN_OK;
}

template <typename T>
static int launch_verify(const T* q, long long Nq, long long q_offset, const T* g, long long Ng, const unsigned long long* claim,
                         const float* block_max, const float* rb_min_d2, unsigned char* beaten, cudaStream_t s) {
  const long long chunks = (Ng + kChunk - 1) / kChunk;
  static DeviceOnce attr_once;
  if (attr_once.first_time())
    HN_CUDA(cudaFuncSetAttribute(mutual_verify_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kVerifySmem)));
  mutual_verify_kernel<T><<<static_cast<unsigned>((chunks + kVerifyWarps - 1) / kVerifyWarps), kVerifyWarps * 32, kVerifySmem, s>>>(
      q, Nq, q_offset, g, Ng, claim, block_max, rb_min_d2, static_cast<int>((Nq + 31) / 32), kVerifyMargin, 1.0f / kDotScale, beaten);
  HN_CUDA(cudaGetLastError());
  count_launch();
  return HN_OK;
}

extern "C" int hn_mutual_verify(const float* q, long long Nq, long long q_offset, const float* g, long long Ng,
                                const unsigned long long* claim, const float* block_max, const float* rb_min_d2,
                                unsigned char* beaten, void* stream) {
  HN_REQUIRE(q && g && claim && block_max && rb_min_d2 && beaten, "hn_mutual_verify: NULL argument");
  HN_REQUIRE(q_offset >= 0, "hn_mutual_verify: q_offset must be >= 0 (got %lld)", q_offset);
  HN_REQUIRE(Nq >= 1 && Ng >= 1 && Nq + q_offset < (1LL << 32), "hn_mutual_verify: size out of range");
  return launch_verify(q, Nq, q_offset, g, Ng, claim, block_max, rb_min_d2, beaten, static_cast<cudaStream_t>(stream));
}

extern "C" long long hn_mutual_workspace_bytes(long long Nq, long long Ng) {
  if (Nq < 0 || Ng < 0) return 0;
  return static_cast<long long>(carve_match(nullptr, Nq, Ng, true).bytes);
}

// hn_match_mutual / hn_match_mutual_typed; fn names the entry point in error messages.
static int mutual_entry(const char* fn, const void* q, const void* g, int desc_dtype, const void* q16, const void* g16, long long Nq,
                        long long Ng, float* d1, float* d2, int32_t* i1, int32_t* i2, unsigned char* mutual, void* workspace,
                        long long workspace_bytes, void* stream) {
  HN_REQUIRE(q && g && d1 && d2 && i1 && mutual && workspace, "%s: NULL argument (d1, d2, i1 and mutual are required outputs)", fn);
  HN_TRY(check_rows(fn, desc_dtype, q, g));
  HN_REQUIRE(workspace_bytes >= hn_mutual_workspace_bytes(Nq, Ng), "%s: workspace too small", fn);
  HN_REQUIRE(Nq >= 1 && Ng >= 1, "%s: empty input (Nq=%lld, Ng=%lld)", fn, Nq, Ng);   // sizes the carve below relies on
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const MatchWs w = carve_match(workspace, Nq, Ng, true);
  HN_TRY(match_entry(fn, q, g, desc_dtype, q16, g16, Nq, Ng, 0, d1, d2, i1, i2, w.block_max, workspace, workspace_bytes, nullptr, stream));
  HN_CUDA(cudaMemsetAsync(w.claim, 0x7f, static_cast<size_t>(Ng) * 8, s));   // "unclaimed"
  HN_CUDA(cudaMemsetAsync(w.beaten, 0, static_cast<size_t>(Ng), s));
  HN_TRY(hn_mutual_claims(i1, d1, d2, Nq, 0, w.claim, Ng, w.rb_min_d2, stream));
  HN_TRY(with_rows(desc_dtype, [&](auto t) -> int {
    using T = decltype(t);
    return launch_verify(static_cast<const T*>(q), Nq, 0, static_cast<const T*>(g), Ng, w.claim, w.block_max, w.rb_min_d2, w.beaten, s);
  }));
  mutual_final_kernel<<<static_cast<unsigned>((Nq + 255) / 256), 256, 0, s>>>(i1, Nq, 0, w.claim, w.beaten, Ng, mutual);
  HN_CUDA(cudaGetLastError());
  count_launch();
  return HN_OK;
}

extern "C" int hn_match_mutual(const float* q, const float* g, const void* q16, const void* g16, long long Nq, long long Ng,
                               float* d1, float* d2, int32_t* i1, int32_t* i2, unsigned char* mutual, void* workspace,
                               long long workspace_bytes, void* stream) {
  return mutual_entry("hn_match_mutual", q, g, HN_F32, q16, g16, Nq, Ng, d1, d2, i1, i2, mutual, workspace, workspace_bytes, stream);
}

extern "C" int hn_match_mutual_typed(const void* q, const void* g, int desc_dtype, const void* q16, const void* g16, long long Nq,
                                     long long Ng, float* d1, float* d2, int32_t* i1, int32_t* i2, unsigned char* mutual,
                                     void* workspace, long long workspace_bytes, void* stream) {
  return mutual_entry("hn_match_mutual_typed", q, g, desc_dtype, q16, g16, Nq, Ng, d1, d2, i1, i2, mutual, workspace, workspace_bytes,
                      stream);
}

// ------------------------------------------------------------------------------------------------------------
// batched matching: B problems in one launch sequence, padded (hn_match_batched) or over row ranges of concatenated sets
// (hn_match_pairs)
// ------------------------------------------------------------------------------------------------------------
// Nq / Ng: the per-pair maxima (output pitch). with_packed: room for B*Nq and B*Ng packed rows in front (hn_match_batched).
// width = kTopKC (hn_match_pairs_topk): lists of kTopKC chunks and their dropped maxima.
static MatchWs carve_batched(void* ws, long long B, long long Nq, long long Ng, bool with_mutual, bool with_packed, int width = kTopC) {
  MatchWs w{};
  char* b = static_cast<char*>(ws);
  size_t off = 0;
  auto take = [&](size_t n) { char* r = b ? b + off : nullptr; off += align256(n); return r; };
  const size_t rows_q = static_cast<size_t>(B) * Nq, rows_g = static_cast<size_t>(B) * Ng;
  w.q16 = with_packed ? take(rows_q * 128 * 2) : nullptr;
  w.g16 = with_packed ? take(rows_g * 128 * 2) : nullptr;
  // candidate lists [rows][segments][width]: a segment holds at least one gallery tile, so at most min(16, tiles) of them
  const size_t lists = rows_q * batched_max_segments(Ng);
  w.cand = reinterpret_cast<int*>(take(lists * width * 4));
  w.cand_val = reinterpret_cast<float*>(take(lists * width * 4));
  if (width == kTopKC) w.cand_drop = reinterpret_cast<float*>(take(lists * 4));
  if (with_mutual) {
    w.block_max = reinterpret_cast<float*>(take(static_cast<size_t>(B) * hn_block_max_elems(Nq, Ng) * 4));
    w.claim = reinterpret_cast<unsigned long long*>(take(rows_g * 8));
    w.beaten = reinterpret_cast<unsigned char*>(take(rows_g));
    w.rb_min_d2 = reinterpret_cast<float*>(take(static_cast<size_t>(B) * ((Nq + 31) / 32) * 4));
  }
  w.bytes = off;
  return w;
}

// Where the pairs of a batched call live. With `pairs` (hn_match_pairs): row ranges [B][4] = (q_start, q_len, g_start, g_len)
// of the concatenated sets of q_rows / g_rows rows. Without (hn_match_batched): the padded layout, pair b at rows b * max_q /
// b * max_g with q_len[b] / g_len[b] valid rows (NULL = all), q_rows = B * max_q, g_rows = B * max_g.
struct PairLayout {
  const int* pairs;
  const int* q_len;
  const int* g_len;
  long long B, max_q, max_g, q_rows, g_rows;
};

// The launch sequence of hn_match_pairs (TABLE) and hn_match_batched: GEMM + shortlist, re-rank, and with `mutual` the column
// side. q16 / g16 are the packed rows of q / g.
// The shortlist GEMM's parameters of a batched call (everything but the segment count): lists of w, operand maps over q16 /
// g16 laid out as L says.
static int pairs_params(bool f8, bool table, const void* q16, const void* g16, const PairLayout& L, const MatchWs& w, DistParams* dp) {
  *dp = shortlist_params(f8, L.max_q, L.max_g, w.cand, w.cand_val, w.block_max);
  // the table form's maps run over the concatenated sets, the padded form's over [B][N] rows
  HN_TRY(make_operand_map(&dp->side[0].tmA, q16, f8, 128, table ? L.q_rows : L.max_q, table ? 0 : L.B, kDistTile));
  HN_TRY(make_operand_map(&dp->side[0].tmB, g16, f8, 128, table ? L.g_rows : L.max_g, table ? 0 : L.B, kDistTile));
  dp->q_len = L.q_len;
  dp->g_len = L.g_len;
  dp->batch = static_cast<int>(L.B);
  dp->pairs = L.pairs;
  dp->q_rows = L.q_rows;
  dp->g_rows = L.g_rows;
  dp->cand_drop = w.cand_drop;
  return HN_OK;
}

template <bool TABLE, typename T>
static int run_pairs(const T* q, const void* q16, const T* g, const void* g16, const PairLayout& L, float* d1,
                     float* d2, int32_t* i1, int32_t* i2, unsigned char* mutual, const MatchWs& w, cudaStream_t s) {
  constexpr bool F8 = kF8Rows<T>;
  int sm = 0;
  HN_TRY(device_sm_count(&sm));
  const long long B = L.B, Nq = L.max_q, Ng = L.max_g, rows_q = B * Nq, rows_g = B * Ng;
  const int threads = 256;
  DistParams dp;
  HN_TRY(pairs_params(F8, TABLE, q16, g16, L, w, &dp));
  {
    MatchTimer timer(1, s);
    // segments from the per-pair maxima (lengths live on the device): B * ceil(Nq / 256) query blocks over a gallery of Ng
    const long long m_blocks = (Nq + 2 * kDistTile - 1) / (2 * kDistTile);
    dp.segments = pick_segments(B * m_blocks * 2 * kDistTile, 2 * kDistTile, Ng, sm, static_cast<int>(batched_max_segments(Ng)));
    const int grid = static_cast<int>(std::min<long long>(B * m_blocks * dp.segments, sm));
    if (TABLE) HN_TRY((launch_dist<2, EPI_SHORTLIST_PAIRS, F8>(dp, grid, 1, s)));
    else HN_TRY((launch_dist<2, EPI_SHORTLIST_BATCHED, F8>(dp, grid, 1, s)));
  }
  {
    MatchTimer timer(2, s);
    rerank_batched_kernel<TABLE, T><<<static_cast<unsigned>((rows_q + 3) / 4), 128, 0, s>>>(
        q, g, w.cand, w.cand_val, kRerankMargin, B, Nq, Ng, L.q_len, L.g_len, dp.segments * kTopC, d1, d2, i1, i2, L.pairs, L.q_rows, L.g_rows);
    HN_CUDA(cudaGetLastError());
    count_launch();
  }
  if (mutual) {
    HN_CUDA(cudaMemsetAsync(w.claim, 0x7f, static_cast<size_t>(rows_g) * 8, s));   // "unclaimed"
    HN_CUDA(cudaMemsetAsync(w.beaten, 0, static_cast<size_t>(rows_g), s));
    const long long nrb = (Nq + 31) / 32, chunks = (Ng + kChunk - 1) / kChunk;
    mutual_claim_batched_kernel<TABLE><<<static_cast<unsigned>((B * nrb * 32 + threads - 1) / threads), threads, 0, s>>>(
        i1, d1, d2, B, Nq, Ng, L.q_len, L.g_len, w.claim, w.rb_min_d2, L.pairs, L.q_rows, L.g_rows);
    static DeviceOnce attr_once;
    if (attr_once.first_time())
      HN_CUDA(cudaFuncSetAttribute(mutual_verify_batched_kernel<TABLE, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kVerifySmem)));
    mutual_verify_batched_kernel<TABLE, T><<<static_cast<unsigned>((B * chunks + kVerifyWarps - 1) / kVerifyWarps), kVerifyWarps * 32, kVerifySmem, s>>>(
        q, g, B, Nq, Ng, L.q_len, L.g_len, w.claim, w.block_max, w.rb_min_d2, kVerifyMargin, 1.0f / kDotScale, w.beaten, L.pairs, L.q_rows,
        L.g_rows);
    mutual_final_batched_kernel<TABLE><<<static_cast<unsigned>((rows_q + threads - 1) / threads), threads, 0, s>>>(
        i1, B, Nq, Ng, L.q_len, L.g_len, w.claim, w.beaten, mutual, L.pairs, L.q_rows, L.g_rows);
    HN_CUDA(cudaGetLastError());
    count_launch(3);
  }
  return HN_OK;
}

extern "C" long long hn_match_batched_workspace_bytes(long long B, long long Nq, long long Ng, int with_mutual) {
  if (B < 0 || Nq < 0 || Ng < 0) return 0;
  return static_cast<long long>(carve_batched(nullptr, B, Nq, Ng, with_mutual != 0, true).bytes);
}

template <typename T>
static int run_batched(const T* q, const T* g, long long B, long long Nq, long long Ng, const int32_t* q_len, const int32_t* g_len,
                       float* d1, float* d2, int32_t* i1, int32_t* i2, unsigned char* mutual, void* workspace, cudaStream_t s) {
  const MatchWs w = carve_batched(workspace, B, Nq, Ng, mutual != nullptr, true);
  const long long rows_q = B * Nq, rows_g = B * Ng;
  {
    MatchTimer timer(0, s);
    launch_pack(q, rows_q, w.q16, 0, s);
    launch_pack(g, rows_g, w.g16, 1, s);
    HN_CUDA(cudaGetLastError());
    count_launch(2);
  }
  const PairLayout L = {nullptr, q_len, g_len, B, Nq, Ng, rows_q, rows_g};
  return run_pairs<false>(q, w.q16, g, w.g16, L, d1, d2, i1, i2, mutual, w, s);
}

// hn_match_batched / hn_match_batched_typed; fn names the entry point in error messages.
static int batched_entry(const char* fn, const void* q, const void* g, int desc_dtype, long long B, long long Nq, long long Ng,
                         const int32_t* q_len, const int32_t* g_len, float* d1, float* d2, int32_t* i1, int32_t* i2,
                         unsigned char* mutual, void* workspace, long long workspace_bytes, void* stream) {
  HN_REQUIRE(q && g && d1 && d2 && i1 && i2 && workspace, "%s: NULL argument (q, g, d1, d2, i1, i2 and workspace are required)", fn);
  HN_TRY(check_rows(fn, desc_dtype, q, g));
  HN_REQUIRE(B >= 1 && Nq >= 1 && Ng >= 1, "%s: empty input (B=%lld, Nq=%lld, Ng=%lld)", fn, B, Nq, Ng);
  HN_REQUIRE(Nq < (1LL << 31) / B && Ng < (1LL << 31) / B, "%s: B*Nq and B*Ng must stay below 2^31 rows", fn);
  HN_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "%s: workspace must be 256-byte aligned", fn);
  HN_REQUIRE(workspace_bytes >= hn_match_batched_workspace_bytes(B, Nq, Ng, mutual != nullptr), "%s: workspace too small", fn);
  return with_rows(desc_dtype, [&](auto t) -> int {
    using T = decltype(t);
    return run_batched(static_cast<const T*>(q), static_cast<const T*>(g), B, Nq, Ng, q_len, g_len, d1, d2, i1, i2, mutual, workspace,
                       static_cast<cudaStream_t>(stream));
  });
}

extern "C" int hn_match_batched(const float* q, const float* g, long long B, long long Nq, long long Ng, const int32_t* q_len,
                                const int32_t* g_len, float* d1, float* d2, int32_t* i1, int32_t* i2, unsigned char* mutual,
                                void* workspace, long long workspace_bytes, void* stream) {
  return batched_entry("hn_match_batched", q, g, HN_F32, B, Nq, Ng, q_len, g_len, d1, d2, i1, i2, mutual, workspace, workspace_bytes,
                       stream);
}

extern "C" int hn_match_batched_typed(const void* q, const void* g, int desc_dtype, long long B, long long Nq, long long Ng,
                                      const int32_t* q_len, const int32_t* g_len, float* d1, float* d2, int32_t* i1, int32_t* i2,
                                      unsigned char* mutual, void* workspace, long long workspace_bytes, void* stream) {
  return batched_entry("hn_match_batched_typed", q, g, desc_dtype, B, Nq, Ng, q_len, g_len, d1, d2, i1, i2, mutual, workspace,
                       workspace_bytes, stream);
}

extern "C" long long hn_match_pairs_workspace_bytes(long long B, long long max_q, long long max_g, int with_mutual) {
  if (B < 0 || max_q < 0 || max_g < 0) return 0;
  return static_cast<long long>(carve_batched(nullptr, B, max_q, max_g, with_mutual != 0, false).bytes);
}

// Argument checks of a pair-table call (hn_match_pairs_typed, hn_match_pairs_topk_typed) up to the workspace size.
static int check_pairs(const char* fn, int desc_dtype, const void* q, const void* q16, long long Nq_rows, const void* g, const void* g16,
                       long long Ng_rows, long long B, long long max_q, long long max_g, const void* workspace) {
  HN_TRY(check_rows(fn, desc_dtype, q, g));
  HN_REQUIRE(B >= 1 && max_q >= 1 && max_g >= 1 && Nq_rows >= 1 && Ng_rows >= 1,
             "%s: empty input (B=%lld, max_q=%lld, max_g=%lld, Nq_rows=%lld, Ng_rows=%lld)", fn, B, max_q, max_g, Nq_rows, Ng_rows);
  HN_REQUIRE(Nq_rows < (1LL << 31) && Ng_rows < (1LL << 31), "%s: a descriptor set has 2^31 rows or more", fn);
  HN_REQUIRE(max_q < (1LL << 31) / B && max_g < (1LL << 31) / B, "%s: B*max_q and B*max_g must stay below 2^31 rows", fn);
  HN_REQUIRE((reinterpret_cast<uintptr_t>(q16) & 15) == 0 && (reinterpret_cast<uintptr_t>(g16) & 15) == 0,
             "%s: packed operands must be 16-byte aligned", fn);
  HN_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "%s: workspace must be 256-byte aligned", fn);
  return HN_OK;
}

// hn_match_pairs / hn_match_pairs_typed; fn names the entry point in error messages.
static int pairs_entry(const char* fn, const void* q, const void* q16, long long Nq_rows, const void* g, const void* g16, long long Ng_rows,
                       int desc_dtype, const int32_t* pairs, long long B, long long max_q, long long max_g, float* d1, float* d2,
                       int32_t* i1, int32_t* i2, unsigned char* mutual, void* workspace, long long workspace_bytes, void* stream) {
  HN_REQUIRE(q && q16 && g && g16 && pairs && d1 && d2 && i1 && i2 && workspace,
             "%s: NULL argument (q, q16, g, g16, pairs, d1, d2, i1, i2 and workspace are required)", fn);
  HN_TRY(check_pairs(fn, desc_dtype, q, q16, Nq_rows, g, g16, Ng_rows, B, max_q, max_g, workspace));
  HN_REQUIRE(workspace_bytes >= hn_match_pairs_workspace_bytes(B, max_q, max_g, mutual != nullptr), "%s: workspace too small", fn);
  const MatchWs w = carve_batched(workspace, B, max_q, max_g, mutual != nullptr, false);
  const PairLayout L = {pairs, nullptr, nullptr, B, max_q, max_g, Nq_rows, Ng_rows};
  return with_rows(desc_dtype, [&](auto t) -> int {
    using T = decltype(t);
    return run_pairs<true>(static_cast<const T*>(q), q16, static_cast<const T*>(g), g16, L, d1, d2, i1, i2, mutual, w,
                           static_cast<cudaStream_t>(stream));
  });
}

extern "C" int hn_match_pairs(const float* q, const void* q16, long long Nq_rows, const float* g, const void* g16, long long Ng_rows,
                              const int32_t* pairs, long long B, long long max_q, long long max_g, float* d1, float* d2, int32_t* i1,
                              int32_t* i2, unsigned char* mutual, void* workspace, long long workspace_bytes, void* stream) {
  return pairs_entry("hn_match_pairs", q, q16, Nq_rows, g, g16, Ng_rows, HN_F32, pairs, B, max_q, max_g, d1, d2, i1, i2, mutual,
                     workspace, workspace_bytes, stream);
}

extern "C" int hn_match_pairs_typed(const void* q, const void* q16, long long Nq_rows, const void* g, const void* g16,
                                    long long Ng_rows, int desc_dtype, const int32_t* pairs, long long B, long long max_q,
                                    long long max_g, float* d1, float* d2, int32_t* i1, int32_t* i2, unsigned char* mutual,
                                    void* workspace, long long workspace_bytes, void* stream) {
  return pairs_entry("hn_match_pairs_typed", q, q16, Nq_rows, g, g16, Ng_rows, desc_dtype, pairs, B, max_q, max_g, d1, d2, i1, i2,
                     mutual, workspace, workspace_bytes, stream);
}

// ---- k nearest neighbours ----------------------------------------------------------------------------------------------

extern "C" long long hn_match_topk_workspace_bytes(long long Nq, long long Ng) {
  if (Nq < 0 || Ng < 0) return 0;
  return static_cast<long long>(carve_match(nullptr, Nq, Ng, false, kTopKC).bytes);
}

extern "C" long long hn_match_pairs_topk_workspace_bytes(long long B, long long max_q, long long max_g) {
  if (B < 0 || max_q < 0 || max_g < 0) return 0;
  return static_cast<long long>(carve_batched(nullptr, B, max_q, max_g, false, false, kTopKC).bytes);
}

// Stages 0 and 1 of hn_match_topk_typed and hn_match_radius_count_typed on validated arguments: packing, then the single-CTA
// GEMM with top-kTopKC lists over batched_max_segments(Ng) (up to kMaxBatchedSegments) segments, so that a list spans at most
// 1/16 of the gallery (the bound on a fallback scan).
template <typename T>
static int run_topk_lists(const T* q, const T* g, const void* q16_in, const void* g16_in, long long Nq, long long Ng, const MatchWs& w,
                          cudaStream_t s) {
  int sm = 0;
  HN_TRY(device_sm_count(&sm));
  constexpr bool F8 = kF8Rows<T>;
  HN_TRY(pack_operands(q, g, q16_in, g16_in, Nq, Ng, w, s));
  DistParams dp = shortlist_params(F8, Nq, Ng, w.cand, w.cand_val, nullptr);
  dp.cand_drop = w.cand_drop;
  HN_TRY(make_operand_map(&dp.side[0].tmA, q16_in ? q16_in : w.q16, F8, 128, Nq, 0, kDistTile));
  HN_TRY(make_operand_map(&dp.side[0].tmB, g16_in ? g16_in : w.g16, F8, 128, Ng, 0, kDistTile));
  dp.segments = static_cast<int>(batched_max_segments(Ng));
  MatchTimer timer(1, s);
  const long long items = ((Nq + 2 * kDistTile - 1) / (2 * kDistTile)) * dp.segments;
  return launch_dist<2, EPI_SHORTLIST, F8, kTopKC>(dp, static_cast<int>(std::min<long long>(items, sm)), 1, s);
}

// The launch sequence of hn_match_topk_typed on validated arguments: the top-k lists, then the re-rank.
template <typename T>
static int run_match_topk(const T* q, const T* g, const void* q16_in, const void* g16_in, long long Nq, long long Ng, int k, float* dist,
                          int32_t* idx, const MatchWs& w, cudaStream_t s) {
  HN_TRY(run_topk_lists(q, g, q16_in, g16_in, Nq, Ng, w, s));
  const int segments = static_cast<int>(batched_max_segments(Ng));
  unsigned long long* fallback_rows = nullptr;
  HN_TRY(topk_fallback_counter(&fallback_rows));
  {
    MatchTimer timer(2, s);
    rerank_topk_kernel<T><<<static_cast<unsigned>((Nq + 3) / 4), 128, 0, s>>>(q, g, w.cand, w.cand_val, w.cand_drop, kRerankMargin, Nq,
                                                                                Ng, segments, k, dist, idx, fallback_rows);
    HN_CUDA(cudaGetLastError());
    count_launch();
  }
  return HN_OK;
}

extern "C" int hn_match_topk_typed(const void* q, const void* g, int desc_dtype, const void* q16, const void* g16, long long Nq,
                                   long long Ng, int k, float* dist, int32_t* idx, void* workspace, long long workspace_bytes,
                                   void* stream) {
  const char* fn = "hn_match_topk_typed";
  HN_REQUIRE(q && g && dist && idx && workspace, "%s: NULL argument (q, g, dist, idx and workspace are required)", fn);
  HN_REQUIRE(k >= 1 && k <= kTopKMax, "%s: k must be in [1, %d] (got %d)", fn, kTopKMax, k);
  HN_TRY(check_match(fn, desc_dtype, q, g, Nq, Ng, 0, workspace));
  HN_REQUIRE(workspace_bytes >= hn_match_topk_workspace_bytes(Nq, Ng), "%s: workspace too small", fn);
  HN_REQUIRE((reinterpret_cast<uintptr_t>(q16) & 15) == 0 && (reinterpret_cast<uintptr_t>(g16) & 15) == 0,
             "%s: packed operands must be 16-byte aligned", fn);
  return with_rows(desc_dtype, [&](auto t) -> int {
    using T = decltype(t);
    return run_match_topk(static_cast<const T*>(q), static_cast<const T*>(g), q16, g16, Nq, Ng, k, dist, idx,
                          carve_match(workspace, Nq, Ng, false, kTopKC), static_cast<cudaStream_t>(stream));
  });
}

// Stage 1 of hn_match_pairs_topk_typed and hn_match_pairs_radius_count_typed on validated arguments: the pair-table GEMM with
// top-kTopKC lists over batched_max_segments(max_g) (up to kMaxBatchedSegments) segments of each pair's gallery.
template <bool F8>
static int run_pairs_topk_lists(const void* q16, const void* g16, const PairLayout& L, const MatchWs& w, cudaStream_t s) {
  int sm = 0;
  HN_TRY(device_sm_count(&sm));
  DistParams dp;
  HN_TRY(pairs_params(F8, true, q16, g16, L, w, &dp));
  dp.segments = static_cast<int>(batched_max_segments(L.max_g));
  MatchTimer timer(1, s);
  const long long m_blocks = (L.max_q + 2 * kDistTile - 1) / (2 * kDistTile);
  const int grid = static_cast<int>(std::min<long long>(L.B * m_blocks * dp.segments, sm));
  return launch_dist<2, EPI_SHORTLIST_PAIRS, F8, kTopKC>(dp, grid, 1, s);
}

// The launch sequence of hn_match_pairs_topk_typed on validated arguments: the top-k lists, then the re-rank.
template <typename T>
static int run_pairs_topk(const T* q, const void* q16, const T* g, const void* g16, const PairLayout& L, int k, float* dist, int32_t* idx,
                          const MatchWs& w, cudaStream_t s) {
  HN_TRY(run_pairs_topk_lists<kF8Rows<T>>(q16, g16, L, w, s));
  const int segments = static_cast<int>(batched_max_segments(L.max_g));
  unsigned long long* fallback_rows = nullptr;
  HN_TRY(topk_fallback_counter(&fallback_rows));
  {
    MatchTimer timer(2, s);
    rerank_topk_pairs_kernel<T><<<static_cast<unsigned>((L.B * L.max_q + 3) / 4), 128, 0, s>>>(
        q, g, w.cand, w.cand_val, w.cand_drop, kRerankMargin, L.B, L.max_q, L.max_g, L.pairs, L.q_rows, L.g_rows, segments, k, dist,
        idx, fallback_rows);
    HN_CUDA(cudaGetLastError());
    count_launch();
  }
  return HN_OK;
}

extern "C" int hn_match_pairs_topk_typed(const void* q, const void* q16, long long Nq_rows, const void* g, const void* g16,
                                         long long Ng_rows, int desc_dtype, const int32_t* pairs, long long B, long long max_q,
                                         long long max_g, int k, float* dist, int32_t* idx, void* workspace, long long workspace_bytes,
                                         void* stream) {
  const char* fn = "hn_match_pairs_topk_typed";
  HN_REQUIRE(q && q16 && g && g16 && pairs && dist && idx && workspace,
             "%s: NULL argument (q, q16, g, g16, pairs, dist, idx and workspace are required)", fn);
  HN_REQUIRE(k >= 1 && k <= kTopKMax, "%s: k must be in [1, %d] (got %d)", fn, kTopKMax, k);
  HN_TRY(check_pairs(fn, desc_dtype, q, q16, Nq_rows, g, g16, Ng_rows, B, max_q, max_g, workspace));
  HN_REQUIRE(workspace_bytes >= hn_match_pairs_topk_workspace_bytes(B, max_q, max_g), "%s: workspace too small", fn);
  const MatchWs w = carve_batched(workspace, B, max_q, max_g, false, false, kTopKC);
  const PairLayout L = {pairs, nullptr, nullptr, B, max_q, max_g, Nq_rows, Ng_rows};
  return with_rows(desc_dtype, [&](auto t) -> int {
    using T = decltype(t);
    return run_pairs_topk(static_cast<const T*>(q), q16, static_cast<const T*>(g), g16, L, k, dist, idx, w,
                          static_cast<cudaStream_t>(stream));
  });
}

// ---- radius matching -----------------------------------------------------------------------------------------------------

// The re-rank threshold of radius r in the GEMM's scaled dot units (see rerank_radius_row): -inf when every column is an entry
// (d <= sqrtf(4) = 2 < r), +inf when none is (d >= sqrtf(1e-8f) >= r; r <= 0 included), else P(r) / kDotScale - kRerankMargin.
static float radius_threshold(float r) {
  if (r > 2.0f) return -INFINITY;
  if (!(r > sqrtf(1e-8f))) return INFINITY;
  const double p = 1.0 - 0.5 * static_cast<double>(r) * static_cast<double>(r) * (1.0 + 0x1p-20);
  return static_cast<float>(p / kDotScale) - kRerankMargin;
}

// Workspace of a radius call: the top-k layout m (carve_match / carve_batched with kTopKC), then the scan's tile sums.
struct RadiusWs {
  MatchWs m;
  long long* tile_sum;
  size_t bytes;
};
static RadiusWs carve_radius(void* ws, const MatchWs& m, long long rows) {
  RadiusWs w{m, ws ? reinterpret_cast<long long*>(static_cast<char*>(ws) + m.bytes) : nullptr, 0};
  w.bytes = m.bytes + align256(static_cast<size_t>((rows + kScanTile - 1) / kScanTile) * 8);
  return w;
}

extern "C" long long hn_match_radius_workspace_bytes(long long Nq, long long Ng) {
  if (Nq < 0 || Ng < 0) return 0;
  return static_cast<long long>(carve_radius(nullptr, carve_match(nullptr, Nq, Ng, false, kTopKC), Nq).bytes);
}

extern "C" long long hn_match_pairs_radius_workspace_bytes(long long B, long long max_q, long long max_g) {
  if (B < 0 || max_q < 0 || max_g < 0) return 0;
  return static_cast<long long>(carve_radius(nullptr, carve_batched(nullptr, B, max_q, max_g, false, false, kTopKC), B * max_q).bytes);
}

// Argument checks shared by the four radius entry points (the count passes capacity 0 and no col / dist).
static int check_radius(const char* fn, float radius, const long long* row_ptr, long long capacity, const int32_t* col, const float* dist) {
  HN_REQUIRE(!std::isnan(radius), "%s: radius is NaN", fn);
  HN_REQUIRE(capacity >= 0, "%s: capacity must be >= 0 (got %lld)", fn, capacity);
  HN_REQUIRE(col || capacity == 0, "%s: col is NULL with capacity %lld > 0", fn, capacity);
  HN_REQUIRE((reinterpret_cast<uintptr_t>(row_ptr) & 7) == 0, "%s: row_ptr must be 8-byte aligned", fn);
  HN_REQUIRE(((reinterpret_cast<uintptr_t>(col) | reinterpret_cast<uintptr_t>(dist)) & 3) == 0, "%s: col and dist must be 4-byte aligned",
             fn);
  return HN_OK;
}

// The count or fill re-rank of a radius call (stage 2) over `rows` rows; the count also turns the counts into row offsets.
template <bool TABLE, bool FILL, typename T>
static int launch_radius(const T* q, const T* g, const RadiusWs& w, float radius, long long rows, long long nq_pad, long long ng_pad,
                         const PairLayout* L, int segments, long long* row_ptr, long long capacity, int32_t* col, float* dist,
                         cudaStream_t s) {
  unsigned long long* fallback_rows = nullptr;
  if (!FILL) HN_TRY(topk_fallback_counter(&fallback_rows));
  MatchTimer timer(2, s);
  rerank_radius_kernel<TABLE, FILL, T><<<static_cast<unsigned>((rows + 3) / 4), 128, 0, s>>>(
      q, g, w.m.cand, w.m.cand_val, w.m.cand_drop, radius_threshold(radius), radius, rows, nq_pad, ng_pad, L ? L->pairs : nullptr,
      L ? L->q_rows : 0, L ? L->g_rows : 0, segments, row_ptr, capacity, col, dist, fallback_rows);
  HN_CUDA(cudaGetLastError());
  count_launch();
  if (!FILL) {
    const unsigned tiles = static_cast<unsigned>((rows + kScanTile - 1) / kScanTile);
    scan_tile_sum_kernel<<<tiles, kScanThreads, 0, s>>>(row_ptr + 1, rows, w.tile_sum);
    scan_tile_offsets_kernel<<<1, kScanThreads, 0, s>>>(w.tile_sum, tiles);
    scan_tile_apply_kernel<<<tiles, kScanThreads, 0, s>>>(row_ptr + 1, rows, w.tile_sum);
    HN_CUDA(cudaGetLastError());
    count_launch(3);
  }
  return HN_OK;
}

// hn_match_radius_count_typed (FILL = false: q16 / g16 may be given) and hn_match_radius_fill_typed.
template <bool FILL>
static int radius_entry(const char* fn, const void* q, const void* g, int desc_dtype, const void* q16, const void* g16, long long Nq,
                        long long Ng, float radius, long long* row_ptr, long long capacity, int32_t* col, float* dist, void* workspace,
                        long long workspace_bytes, void* stream) {
  HN_REQUIRE(q && g && row_ptr && workspace, "%s: NULL argument (q, g, row_ptr and workspace are required)", fn);
  HN_TRY(check_radius(fn, radius, row_ptr, capacity, col, dist));
  HN_TRY(check_match(fn, desc_dtype, q, g, Nq, Ng, 0, workspace));
  HN_REQUIRE(workspace_bytes >= hn_match_radius_workspace_bytes(Nq, Ng), "%s: workspace too small", fn);
  HN_REQUIRE((reinterpret_cast<uintptr_t>(q16) & 15) == 0 && (reinterpret_cast<uintptr_t>(g16) & 15) == 0,
             "%s: packed operands must be 16-byte aligned", fn);
  const RadiusWs w = carve_radius(workspace, carve_match(workspace, Nq, Ng, false, kTopKC), Nq);
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int segments = static_cast<int>(batched_max_segments(Ng));
  return with_rows(desc_dtype, [&](auto t) -> int {
    using T = decltype(t);
    const T *qt = static_cast<const T*>(q), *gt = static_cast<const T*>(g);
    if (!FILL) HN_TRY(run_topk_lists(qt, gt, q16, g16, Nq, Ng, w.m, s));
    return launch_radius<false, FILL>(qt, gt, w, radius, Nq, Nq, Ng, nullptr, segments, row_ptr, capacity, col, dist, s);
  });
}

extern "C" int hn_match_radius_count_typed(const void* q, const void* g, int desc_dtype, const void* q16, const void* g16, long long Nq,
                                           long long Ng, float radius, long long* row_ptr, void* workspace, long long workspace_bytes,
                                           void* stream) {
  return radius_entry<false>("hn_match_radius_count_typed", q, g, desc_dtype, q16, g16, Nq, Ng, radius, row_ptr, 0, nullptr, nullptr,
                             workspace, workspace_bytes, stream);
}

extern "C" int hn_match_radius_fill_typed(const void* q, const void* g, int desc_dtype, long long Nq, long long Ng, float radius,
                                          const long long* row_ptr, long long capacity, int32_t* col, float* dist, void* workspace,
                                          long long workspace_bytes, void* stream) {
  return radius_entry<true>("hn_match_radius_fill_typed", q, g, desc_dtype, nullptr, nullptr, Nq, Ng, radius,
                            const_cast<long long*>(row_ptr), capacity, col, dist, workspace, workspace_bytes, stream);
}

// hn_match_pairs_radius_count_typed and hn_match_pairs_radius_fill_typed.
template <bool FILL>
static int pairs_radius_entry(const char* fn, const void* q, const void* q16, long long Nq_rows, const void* g, const void* g16,
                              long long Ng_rows, int desc_dtype, const int32_t* pairs, long long B, long long max_q, long long max_g,
                              float radius, long long* row_ptr, long long capacity, int32_t* col, float* dist, void* workspace,
                              long long workspace_bytes, void* stream) {
  HN_REQUIRE(q && q16 && g && g16 && pairs && row_ptr && workspace,
             "%s: NULL argument (q, q16, g, g16, pairs, row_ptr and workspace are required)", fn);
  HN_TRY(check_radius(fn, radius, row_ptr, capacity, col, dist));
  HN_TRY(check_pairs(fn, desc_dtype, q, q16, Nq_rows, g, g16, Ng_rows, B, max_q, max_g, workspace));
  HN_REQUIRE(workspace_bytes >= hn_match_pairs_radius_workspace_bytes(B, max_q, max_g), "%s: workspace too small", fn);
  const RadiusWs w = carve_radius(workspace, carve_batched(workspace, B, max_q, max_g, false, false, kTopKC), B * max_q);
  const PairLayout L = {pairs, nullptr, nullptr, B, max_q, max_g, Nq_rows, Ng_rows};
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int segments = static_cast<int>(batched_max_segments(max_g));
  return with_rows(desc_dtype, [&](auto t) -> int {
    using T = decltype(t);
    if (!FILL) HN_TRY(run_pairs_topk_lists<kF8Rows<T>>(q16, g16, L, w.m, s));
    return launch_radius<true, FILL>(static_cast<const T*>(q), static_cast<const T*>(g), w, radius, B * max_q, max_q, max_g, &L, segments,
                                     row_ptr, capacity, col, dist, s);
  });
}

extern "C" int hn_match_pairs_radius_count_typed(const void* q, const void* q16, long long Nq_rows, const void* g, const void* g16,
                                                 long long Ng_rows, int desc_dtype, const int32_t* pairs, long long B, long long max_q,
                                                 long long max_g, float radius, long long* row_ptr, void* workspace,
                                                 long long workspace_bytes, void* stream) {
  return pairs_radius_entry<false>("hn_match_pairs_radius_count_typed", q, q16, Nq_rows, g, g16, Ng_rows, desc_dtype, pairs, B, max_q,
                                   max_g, radius, row_ptr, 0, nullptr, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int hn_match_pairs_radius_fill_typed(const void* q, const void* q16, long long Nq_rows, const void* g, const void* g16,
                                                long long Ng_rows, int desc_dtype, const int32_t* pairs, long long B, long long max_q,
                                                long long max_g, float radius, const long long* row_ptr, long long capacity,
                                                int32_t* col, float* dist, void* workspace, long long workspace_bytes, void* stream) {
  return pairs_radius_entry<true>("hn_match_pairs_radius_fill_typed", q, q16, Nq_rows, g, g16, Ng_rows, desc_dtype, pairs, B, max_q,
                                  max_g, radius, const_cast<long long*>(row_ptr), capacity, col, dist, workspace, workspace_bytes, stream);
}

extern "C" int hn_match_force_kernel(int mode) {
  HN_REQUIRE(mode >= -1 && mode <= 1, "hn_match_force_kernel: mode must be -1 (by size), 0 (single CTA) or 1 (CTA pair)");
  match_kernel_mode() = mode;
  return HN_OK;
}

extern "C" int hn_match_profile_enable(int on) {
  g_match_profile.on = on != 0;
  for (size_t& u : g_match_profile.used) u = 0;
  return HN_OK;
}

extern "C" int hn_match_topk_fallback_enable(int on) {
  if (g_topk_fallback_rows) HN_CUDA(cudaFree(g_topk_fallback_rows));
  g_topk_fallback_rows = nullptr;
  if (on) {
    HN_CUDA(cudaMalloc(&g_topk_fallback_rows, sizeof(unsigned long long)));
    HN_CUDA(cudaMemset(g_topk_fallback_rows, 0, sizeof(unsigned long long)));
  }
  return HN_OK;
}

extern "C" int hn_match_topk_fallback_read(long long* rows_out) {
  HN_REQUIRE(rows_out, "hn_match_topk_fallback_read: NULL argument");
  HN_REQUIRE(g_topk_fallback_rows, "hn_match_topk_fallback_read: the count is not enabled (hn_match_topk_fallback_enable(1))");
  unsigned long long v = 0;
  HN_CUDA(cudaMemcpy(&v, g_topk_fallback_rows, sizeof(v), cudaMemcpyDeviceToHost));
  *rows_out = static_cast<long long>(v);
  HN_CUDA(cudaMemset(g_topk_fallback_rows, 0, sizeof(unsigned long long)));
  return HN_OK;
}

extern "C" int hn_match_profile_read(double ms_out[3], long long launches_out[3]) {
  HN_REQUIRE(ms_out && launches_out, "hn_match_profile_read: NULL argument");
  for (int st = 0; st < 3; ++st) {
    double total = 0.0;
    const size_t pairs = g_match_profile.used[st] / 2;
    for (size_t i = 0; i < pairs; ++i) {
      HN_CUDA(cudaEventSynchronize(g_match_profile.ev[st][2 * i + 1]));
      float ms = 0.f;
      HN_CUDA(cudaEventElapsedTime(&ms, g_match_profile.ev[st][2 * i], g_match_profile.ev[st][2 * i + 1]));
      total += ms;
    }
    ms_out[st] = total;
    launches_out[st] = static_cast<long long>(pairs);
    g_match_profile.used[st] = 0;
  }
  return HN_OK;
}
