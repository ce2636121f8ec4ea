// Fused descriptor-distance kernels: a tcgen05 GEMM (D = A * B^T over 128-d descriptors) whose epilogue
// reduces each 128 x 128 accumulator tile in registers, so the Na x Nb distance matrix never exists in
// HBM. Replaces distance_matrix_vector + the masking / min / sort sequences of the reference
// (hardnet/Losses.py:5-13,95-108; FDLNet-master/utils/math_utils.py:8-19, eval_utils.py:113-114,168-175).
//
// A work item is (block of MB*128 A-rows, segment of B). The A block stays resident in shared memory
// (K <= 384), B tiles of 128 rows stream through a TMA ring, accumulators are double buffered in TMEM.
//
//   EPI_EXACT : operands are 3-way split fp16 (K = 384: hi*hi + hi*lo + lo*hi ~ fp32 dot). Every element
//               goes through the reference arithmetic (norms, eps, sqrt, diagonal / duplicate masks) and
//               feeds a per-row (value, index) minimum. Used for the loss and for hn_dist_min.
//   EPI_SHORTLIST : single fp16 pass (K = 128). Per row, the TOPC best 8-column chunks by dot product
//               are kept (max3 trees + a rarely taken sorted insert); a tiny fp32 kernel then re-ranks
//               those candidates exactly. Used for bulk matching.
//   EPI_SHORTLIST_BATCHED : EPI_SHORTLIST over B independent padded problems (hn_match_batched). Operands are 3-D tensor maps
//               {K, N, B} whose boxes never cross into the next pair (TMA zero-fills past N); a work item is (pair, query block,
//               segment), and each pair has its own row / column counts (q_len / g_len). The batch logic is confined to the
//               item decode, the TMA coordinates, the per-pair bounds and the output offsets, and compiles away elsewhere.
//   EPI_SHORTLIST_PAIRS : the same over row ranges of concatenated sets (hn_match_pairs): pair b's (start, length) per side comes
//               from a device table (table_span), operands are 2-D tensor maps over the concatenated rows and the TMA row
//               coordinate is start + local row. A box may reach past a pair's range into other rows (or past the set, where
//               TMA zero-fills); the per-pair bounds above keep them out: columns past the length are masked to -inf, rows
//               past it are neither stored nor part of the cell maxima. A separate instantiation rather than the padded
//               case of one accessor: reading the padded layout through the table accessor made hn_match_batched 1-2 %
//               slower (DESIGN.md section 5).
//
// F8: the shortlist kernels on e4m3 operand rows (matching on HN_F8E4M3 rows, dist.cu). A K = 128 e4m3 row is 128 bytes, one
// 128B-swizzle atom, so an fp8 operand is the fp16 case with k_blocks = 1: the same shared-memory blocks, tensor maps with the
// same box in bytes, the same descriptor steps; only the MMA kind changes (umma_f8_w, kind::f8f6f4, K = 32 per MMA).
#pragma once

#include "../../include/hardnet_b200.h"
#include "common.cuh"

namespace hn {

constexpr int kDistTile = 128;
constexpr int kDistStages = 4;
constexpr int kTopC = 4;     // chunks kept per row and segment
constexpr int kTopKC = 8;    // the same for the k-nearest-neighbour lists (hn_match_topk), which also keep a dropped maximum
constexpr int kChunk = 8;    // columns per chunk

enum : int { EPI_EXACT = 0, EPI_SHORTLIST = 1, EPI_EXACT_NEI = 2, EPI_SHORTLIST_BATCHED = 3, EPI_SHORTLIST_PAIRS = 4 };   // EXACT_NEI = EXACT + the keypoint-neighbour masks

struct DistSide {
  CUtensorMap tmA;             // rows of this launch direction, [Na, K] 16-bit (e4m3 in the F8 kernels)
  CUtensorMap tmB;             // columns, [Nb, K]
  const float* norm_a;         // |a_i|^2 (hardnet form)
  const float* norm_b;
  unsigned long long* row_pack;  // EXACT: packed (float bits << 32 | col) running minimum per row
  float* pos;                  // EXACT: diagonal distance before masking (may be null)
  int* cand;                   // SHORTLIST: [Na, segments, kTopC] chunk ids
  float* cand_val;             // SHORTLIST: the chunks' approximate (fp16-operand, scaled) dot-product maxima
  float* block_max;            // SHORTLIST, optional: [ceil(Nb / 8)][ceil(Na / 32)] maxima of the approximate dot products over
                               // (32-row block, 8-column chunk) cells: what the column side of mutual NN needs from this GEMM
  int n_row_blocks;            // ceil(Na / 32)
  // neighbour mask (FDLNet-master/latency/rfnet/model/rf_des.py:72-86): (x, y) keypoint coordinates of the row / column items
  // in the anchor image (xy_a*) and in the positive image (xy_p*); a pair closer than nei_c pixels in either gets +10 each
  const float2* xy_a_rows; const float2* xy_a_cols;
  const float2* xy_p_rows; const float2* xy_p_cols;
  long long Na, Nb;
};

struct DistParams {
  DistSide side[2];            // [1] = transposed problem (anchor swap / column minima)
  int k_blocks;                // 128-byte K blocks per row: K / 64 (16-bit operands), 1 (e4m3 operands)
  int segments;
  int form;                    // HN_FORM_*
  int loss_mask;               // apply +1e-8, diagonal +10, (<0.008) +10
  int nei_mask;                // diagonal +10 and the neighbour masks (no +1e-8, no duplicate mask): HardNetNeiMask.loss
  float nei_c;                 // neighbour radius C in pixels
  float dot_scale;             // undoes the power-of-two operand scaling
  // EPI_SHORTLIST_BATCHED only (appended: no parameter of the other kernels moves). side[0].Na / Nb are the padded per-pair
  // sizes, cand / cand_val hold [batch * Na] rows, block_max is [batch][ceil(Nb / 8)][ceil(Na / 32)].
  const int* q_len;            // [batch] valid query rows per pair (NULL = all), clamped to [0, Na]
  const int* g_len;            // [batch] valid gallery rows per pair (NULL = all), clamped to [0, Nb]
  int batch;
  // EPI_SHORTLIST_PAIRS only: [batch][4] = (q_start, q_len, g_start, g_len) and the rows of the concatenated sets (q_len / g_len
  // unused; side[0].Na / Nb are the per-pair maxima max_q / max_g)
  const int* pairs;
  long long q_rows, g_rows;
  // TOPC = kTopKC lists only (appended like the batch fields): [lists] the largest approximate chunk maximum of each list that
  // did not make it (-inf when every chunk of the list was kept)
  float* cand_drop;
};

template <int MB>
constexpr size_t dist_smem_bytes(int k_blocks) {
  return size_t(MB) * k_blocks * (kDistTile * 128) + size_t(kDistStages) * (kDistTile * 128) + 1024 + 256 + 2 * kDistTile * 4 +
         2 * kDistTile * 16 /* column keypoints of the neighbour mask */;
}

// Valid rows of pair b of a padded batch: len[b] clamped to [0, n], or n when no lengths are given.
__device__ __forceinline__ long long pair_len(const int* len, long long b, long long n) {
  return len ? min(max(static_cast<long long>(len[b]), 0ll), n) : n;
}

// One side (0 = query, 1 = gallery) of pair b of a pair table [B][4] = (q_start, q_len, g_start, g_len): the start clamped to
// [0, rows], the length to [0, min(max_len, rows - start)].
struct Span {
  long long start, len;
};
__device__ __forceinline__ Span table_span(const int* pairs, long long b, int side, long long max_len, long long rows) {
  const long long start = min(max(static_cast<long long>(pairs[4 * b + 2 * side]), 0ll), rows);
  return {start, min(max(static_cast<long long>(pairs[4 * b + 2 * side + 1]), 0ll), min(max_len, rows - start))};
}

__device__ __forceinline__ float max3(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }

// c[0..7]: this lane's (= this row's) maxima over eight consecutive 8-column chunks. Returns, in every lane, the maximum over
// the warp's 32 rows of chunk (lane >> 2): a halving butterfly - each exchange keeps half of the chunks and sends the other
// half, so the 8 x 32 values cost 4 + 2 + 1 + 1 + 1 = 9 shuffles instead of 40.
__device__ __forceinline__ float warp_chunk_max8(const float (&c)[8], int lane) {
  const bool b4 = (lane & 16) != 0, b3 = (lane & 8) != 0, b2 = (lane & 4) != 0;
  float a[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const float keep = b4 ? c[t + 4] : c[t], send = b4 ? c[t] : c[t + 4];
    a[t] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 16));
  }
  float b[2];
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const float keep = b3 ? a[t + 2] : a[t], send = b3 ? a[t] : a[t + 2];
    b[t] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 8));
  }
  const float keep = b2 ? b[1] : b[0], send = b2 ? b[0] : b[1];
  float v = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 4));
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return v;
}

// A row's candidate list (one segment; in the CTA-pair kernel one 64-column half of it) at list index `list` of cand /
// cand_val: the C chunk ids (C = kTopC or kTopKC), -1 in unused slots (a segment with fewer than C chunks), and the chunks'
// maxima.
template <int C>
__device__ __forceinline__ void store_cand_list(int* cand, float* cand_val, long long list, const float (&tb)[C], const int (&tc)[C]) {
  static_assert(C % 4 == 0, "lists are stored in 16-byte pieces");
#pragma unroll
  for (int h = 0; h < C; h += 4) {
    *reinterpret_cast<int4*>(cand + list * C + h) = make_int4(tb[h] > -3.0e38f ? tc[h] : -1, tb[h + 1] > -3.0e38f ? tc[h + 1] : -1,
                                                              tb[h + 2] > -3.0e38f ? tc[h + 2] : -1, tb[h + 3] > -3.0e38f ? tc[h + 3] : -1);
    *reinterpret_cast<float4*>(cand_val + list * C + h) = make_float4(tb[h], tb[h + 1], tb[h + 2], tb[h + 3]);
  }
}

// Epilogue warps per accumulator lane quarter. The exact epilogues (loss kernels) cost ~80 instructions per column and a loss-sized
// problem (N = 1024) gives every CTA exactly ONE 128 x 128 tile: with one warp per quarter a thread walked 128 columns alone
// (~10 k dependent instructions = 13 us of a 28 us kernel). Four warps per quarter take 32 columns each and merge through the
// packed atomicMin the segments already use.
template <int EPI>
constexpr int dist_col_split() { return (EPI == EPI_EXACT || EPI == EPI_EXACT_NEI) ? 4 : 1; }

// TOPC: chunks per candidate list of the shortlist epilogues. kTopC for hn_match and its batched forms; kTopKC for the k-nearest-
// neighbour lists, which also record each list's dropped maximum (p.cand_drop) so that the re-rank can tell when a list may
// hide one of the k nearest columns (rerank_topk_row).
template <int MB, int EPI, bool F8 = false, int TOPC = kTopC>
__global__ void __launch_bounds__(64 + 128 * MB * dist_col_split<EPI>(), 1) dist_kernel(const __grid_constant__ DistParams p) {
  constexpr bool EXACT = EPI == EPI_EXACT || EPI == EPI_EXACT_NEI;
  constexpr int CS = dist_col_split<EPI>();
  static_assert(CS == 1 || MB == 1, "the column split is for the single-M-block loss kernels");
  constexpr bool NEI = EPI == EPI_EXACT_NEI;   // compile-time: the plain loss kernel carries none of the mask code
  constexpr bool PAIRS = EPI == EPI_SHORTLIST_PAIRS;
  constexpr bool BATCHED = EPI == EPI_SHORTLIST_BATCHED || PAIRS;
  constexpr bool SHORTLIST = EPI == EPI_SHORTLIST || BATCHED;
  static_assert(!F8 || (SHORTLIST && MB == 2), "e4m3 operands are for the matching GEMMs");
  constexpr bool DROP = TOPC == kTopKC;
  static_assert(TOPC == kTopC || (DROP && (EPI == EPI_SHORTLIST || EPI == EPI_SHORTLIST_PAIRS)), "top-k lists: single problems and pair tables");
  constexpr uint32_t BLK_BYTES = kDistTile * 128;  // 128 rows x 64 fp16 (F8: x 128 e4m3)
  constexpr uint32_t TMEM_COLS = 2 * MB * kDistTile;
  const DistSide& sd = p.side[blockIdx.y];

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  const uint32_t a_base = base;
  const uint32_t b_base = base + MB * p.k_blocks * BLK_BYTES;
  const uint32_t bar_base = b_base + kDistStages * BLK_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kDistStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * kDistStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * kDistStages + 2 + a); };
  const uint32_t afull_bar = bar_base + 8u * (2 * kDistStages + 4);
  const uint32_t aempty_bar = bar_base + 8u * (2 * kDistStages + 5);
  const uint32_t tmem_slot = bar_base + 8u * (2 * kDistStages + 6);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw_addr));
  float* s_nb = reinterpret_cast<float*>(smem_raw + (bar_base + 256u - raw_addr));  // [2][128]
  float4* s_xy = reinterpret_cast<float4*>(smem_raw + (bar_base + 256u + 2 * kDistTile * 4 - raw_addr));  // [2][128] (ax, ay, px, py)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const int m_blocks = static_cast<int>((sd.Na + MB * kDistTile - 1) / (MB * kDistTile));
  const int n_tiles = static_cast<int>((sd.Nb + kDistTile - 1) / kDistTile);
  const int num_items = m_blocks * p.segments * (BATCHED ? p.batch : 1);
  // An item is (pair, query block, segment); a single problem is pair 0. The valid query rows / gallery columns of a pair come
  // from its lengths: producer, issuer and epilogue read the same ones, so they agree on which items and tiles exist.
  auto pair_of = [&](int item) { return BATCHED ? item / (m_blocks * p.segments) : 0; };
  auto pair_rows = [&](int pair) {
    return PAIRS ? table_span(p.pairs, pair, 0, sd.Na, p.q_rows).len : BATCHED ? pair_len(p.q_len, pair, sd.Na) : sd.Na;
  };
  auto pair_cols = [&](int pair) {
    return PAIRS ? table_span(p.pairs, pair, 1, sd.Nb, p.g_rows).len : BATCHED ? pair_len(p.g_len, pair, sd.Nb) : sd.Nb;
  };
  auto pair_tiles = [&](int pair) { return BATCHED ? static_cast<int>((pair_cols(pair) + kDistTile - 1) / kDistTile) : n_tiles; };
  auto seg_range = [&](int seg, int tiles, int& t0, int& t1) {
    t0 = static_cast<int>(static_cast<long long>(tiles) * seg / p.segments);
    t1 = static_cast<int>(static_cast<long long>(tiles) * (seg + 1) / p.segments);
  };

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&sd.tmA);
    tma_prefetch_desc(&sd.tmB);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < kDistStages; ++s) {
        mbar_init(full_bar(s), 1);
        mbar_init(empty_bar(s), 1);
      }
      for (int a = 0; a < 2; ++a) {
        mbar_init(tfull_bar(a), 1);
        mbar_init(tempty_bar(a), 4 * MB * CS);
      }
      mbar_init(afull_bar, 1);
      mbar_init(aempty_bar, 1);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ============================== TMA producer (warp-uniform) ==============================
    {
      int stage = 0;
      uint32_t phase = 0, a_phase = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
        const int pair = pair_of(item), local = item - pair * (m_blocks * p.segments);
        const int mblk = local / p.segments, seg = local - mblk * p.segments;
        int t0, t1;
        int q0 = 0, g0 = 0;   // PAIRS: first row of the pair in each concatenated set; TMA row coordinate = start + local row
        if constexpr (PAIRS) {   // each span read once (the issuer and epilogue need only the lengths)
          const Span qsp = table_span(p.pairs, pair, 0, sd.Na, p.q_rows), gsp = table_span(p.pairs, pair, 1, sd.Nb, p.g_rows);
          seg_range(seg, static_cast<int>((gsp.len + kDistTile - 1) / kDistTile), t0, t1);
          if (static_cast<long long>(mblk) * MB * kDistTile >= qsp.len || t0 == t1) continue;   // as the issuer
          q0 = static_cast<int>(qsp.start);
          g0 = static_cast<int>(gsp.start);
        } else {
          seg_range(seg, pair_tiles(pair), t0, t1);
          if (BATCHED && (static_cast<long long>(mblk) * MB * kDistTile >= pair_rows(pair) || t0 == t1)) continue;   // as the issuer
        }
        mbar_wait(aempty_bar, a_phase ^ 1u);
        if (elect_one()) {
          mbar_arrive_expect_tx(afull_bar, MB * p.k_blocks * BLK_BYTES);
          for (int mb = 0; mb < MB; ++mb)
            for (int kb = 0; kb < p.k_blocks; ++kb) {
              if (PAIRS)
                tma_load_2d(a_base + (mb * p.k_blocks + kb) * BLK_BYTES, &sd.tmA, afull_bar, kb * 64, q0 + (mblk * MB + mb) * kDistTile);
              else if (BATCHED)
                tma_load_3d(a_base + (mb * p.k_blocks + kb) * BLK_BYTES, &sd.tmA, afull_bar, kb * 64, (mblk * MB + mb) * kDistTile, pair);
              else
                tma_load_2d(a_base + (mb * p.k_blocks + kb) * BLK_BYTES, &sd.tmA, afull_bar, kb * 64,
                            (mblk * MB + mb) * kDistTile);
            }
        }
        __syncwarp();
        a_phase ^= 1u;
        for (int t = t0; t < t1; ++t) {
          for (int kb = 0; kb < p.k_blocks; ++kb) {
            mbar_wait(empty_bar(stage), phase ^ 1u);
            if (elect_one()) {
              mbar_arrive_expect_tx(full_bar(stage), BLK_BYTES);
              if (PAIRS) tma_load_2d(b_base + stage * BLK_BYTES, &sd.tmB, full_bar(stage), kb * 64, g0 + t * kDistTile);
              else if (BATCHED) tma_load_3d(b_base + stage * BLK_BYTES, &sd.tmB, full_bar(stage), kb * 64, t * kDistTile, pair);
              else tma_load_2d(b_base + stage * BLK_BYTES, &sd.tmB, full_bar(stage), kb * 64, t * kDistTile);
            }
            __syncwarp();
            if (++stage == kDistStages) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ============================== UMMA issuer (warp-uniform) ==============================
    // Every lane runs the control flow, elect.sync picks the issuing lane; descriptors advance by adding to their lo word.
    {
      const uint32_t idesc = make_idesc_f16(kDistTile, kDistTile, 0);
      constexpr uint32_t HI = kmajor_desc_hi(128);
      const uint32_t a_lo0 = kmajor_desc_lo(a_base);
      const uint32_t b_lo0 = kmajor_desc_lo(b_base);
      int stage = 0;
      uint32_t phase = 0, a_phase = 0;
      int it = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
        const int pair = pair_of(item), local = item - pair * (m_blocks * p.segments);
        const int mblk = local / p.segments, seg = local - mblk * p.segments;
        int t0, t1;
        seg_range(seg, pair_tiles(pair), t0, t1);
        if (BATCHED && (static_cast<long long>(mblk) * MB * kDistTile >= pair_rows(pair) || t0 == t1)) continue;   // as the producer
        mbar_wait(afull_bar, a_phase);
        a_phase ^= 1u;
        tc_fence_after();
        for (int t = t0; t < t1; ++t, ++it) {
          const int acc = it & 1;
          const uint32_t acc_phase = (it >> 1) & 1;
          mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
          tc_fence_after();
          for (int kb = 0; kb < p.k_blocks; ++kb) {
            mbar_wait(full_bar(stage), phase);
            tc_fence_after();
            if (elect_one()) {
              const uint32_t b_lo = b_lo0 + static_cast<uint32_t>(stage) * (BLK_BYTES >> 4);
#pragma unroll
              for (int mb = 0; mb < MB; ++mb) {
                const uint32_t a_lo = a_lo0 + static_cast<uint32_t>(mb * p.k_blocks + kb) * (BLK_BYTES >> 4);
                const uint32_t d_tmem = tmem_base + (acc * MB + mb) * kDistTile;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  if constexpr (F8) umma_f8_w(d_tmem, a_lo + 2u * k, HI, b_lo + 2u * k, HI, idesc, (kb | k) != 0);
                  else umma_f16_w(d_tmem, a_lo + 2u * k, HI, b_lo + 2u * k, HI, idesc, (kb | k) != 0);
                }
              }
              umma_commit(empty_bar(stage));
              if (kb == p.k_blocks - 1) umma_commit(tfull_bar(acc));
            }
            __syncwarp();
            if (++stage == kDistStages) { stage = 0; phase ^= 1u; }
          }
        }
        if (elect_one()) umma_commit(aempty_bar);  // the resident A block may be overwritten once these MMAs retired
        __syncwarp();
      }
    }
  } else {
    // ============================== epilogue ==============================
    const int q = warp & 3;
    const int mb = CS == 1 ? (warp - 2) >> 2 : 0;
    const int cs = CS == 1 ? 0 : (warp - 2) >> 2;   // which 32 of the tile's 128 columns (exact epilogues)
    const int ep_tid = threadIdx.x - 64;  // 0 .. 128*MB*CS-1
    int it = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
      const int pair = pair_of(item), local = item - pair * (m_blocks * p.segments);
      const int mblk = local / p.segments, seg = local - mblk * p.segments;
      // a single problem reads sd.Na / sd.Nb where it uses them
      // 32-bit per-pair bounds (B * Na, B * Nb < 2^31): the epilogue runs at the register limit
      const int rows_b = BATCHED ? static_cast<int>(pair_rows(pair)) : 0, cols_b = BATCHED ? static_cast<int>(pair_cols(pair)) : 0;
      auto rows = [&] { return BATCHED ? static_cast<long long>(rows_b) : sd.Na; };
      auto cols = [&] { return BATCHED ? static_cast<long long>(cols_b) : sd.Nb; };
      int t0, t1;
      seg_range(seg, pair_tiles(pair), t0, t1);
      // a block without valid rows has no tiles in any role; an empty segment (t0 == t1) has none either, but its rows still
      // get their (empty) candidate lists
      if (BATCHED && static_cast<long long>(mblk) * MB * kDistTile >= rows()) continue;
      const long long row = static_cast<long long>(mblk * MB + mb) * kDistTile + q * 32 + lane;
      const bool row_ok = row < rows();

      // per-row running state
      float best = __int_as_float(0x7f800000);
      int best_col = 0x7fffffff;
      float na = 0.f;
      float tb[TOPC];
      int tc[TOPC];
      float drop = -__int_as_float(0x7f800000);   // DROP only
      float2 r_axy = make_float2(0.f, 0.f), r_pxy = make_float2(0.f, 0.f);
      if (EXACT) {
        if (p.form == HN_FORM_HARDNET && row_ok) na = sd.norm_a[row];
        if (NEI && row_ok) { r_axy = sd.xy_a_rows[row]; r_pxy = sd.xy_p_rows[row]; }
      } else {
#pragma unroll
        for (int i = 0; i < TOPC; ++i) { tb[i] = -__int_as_float(0x7f800000); tc[i] = 0; }
      }

      for (int t = t0; t < t1; ++t, ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        const long long col0 = static_cast<long long>(t) * kDistTile;
        if (EXACT && p.form == HN_FORM_HARDNET) {
          // column norms of this tile -> smem (double buffered with the accumulator)
          if (ep_tid < kDistTile) {
            const long long c = col0 + ep_tid;
            s_nb[acc * kDistTile + ep_tid] = c < sd.Nb ? sd.norm_b[c] : 0.f;
          }
          asm volatile("bar.sync 1, %0;" ::"n"(128 * MB * CS) : "memory");
        }
        if (NEI) {
          if (ep_tid < kDistTile) {
            const long long c = col0 + ep_tid;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (c < sd.Nb) { const float2 a = sd.xy_a_cols[c], b = sd.xy_p_cols[c]; v = make_float4(a.x, a.y, b.x, b.y); }
            s_xy[acc * kDistTile + ep_tid] = v;
          }
          asm volatile("bar.sync 1, %0;" ::"n"(128 * MB * CS) : "memory");
        }
        mbar_wait(tfull_bar(acc), acc_phase);
        tc_fence_after();
        const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + (acc * MB + mb) * kDistTile;
        if (SHORTLIST) {
          const bool ragged = col0 + kDistTile > cols();
          // all four TMEM loads are issued before the single wait: one exposed round trip per tile instead of four. The top-k
          // lists (DROP) hold 8 + 8 more registers; there two loads per wait keep the epilogue clear of spills.
          constexpr int LDS = DROP ? 2 : 4;
          float cm[16];   // this row's maxima of the tile's sixteen chunks
#pragma unroll
          for (int h = 0; h < 4; h += LDS) {
            uint32_t r[LDS][32];
#pragma unroll
            for (int gq = 0; gq < LDS; ++gq) tmem_ld32(t_row + (h + gq) * 32, r[gq]);
            tmem_ld_wait();
#pragma unroll
            for (int gq = h; gq < h + LDS; ++gq) {
              const int c0 = gq * 32;
              float v[32];
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[gq - h][j]);
              if (ragged) {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                  if (col0 + c0 + j >= cols()) v[j] = -__int_as_float(0x7f800000);
              }
#pragma unroll
              for (int s = 0; s < 32 / kChunk; ++s) {
                const float* w = v + s * kChunk;
                const float m = fmaxf(max3(w[0], w[1], w[2]), max3(max3(w[3], w[4], w[5]), w[6], w[7]));
                cm[gq * 4 + s] = BATCHED && !row_ok ? -__int_as_float(0x7f800000) : m;   // padding rows stay out of the block maxima
                // the chunk that leaves the list, this one or the evicted last entry, is the smaller of the two
                if constexpr (DROP) drop = fmaxf(drop, fminf(m, tb[TOPC - 1]));
                if (m > tb[TOPC - 1]) {
                  const int id = static_cast<int>((col0 + c0) / kChunk) + s;
                  // sorted insert (descending); strict '>' keeps the earlier chunk on ties
                  if constexpr (TOPC == kTopC) {   // hn_match's lists, written out: the loop below compiles differently
                    const bool g0 = m > tb[0], g1 = m > tb[1], g2 = m > tb[2];
                    tb[3] = g2 ? tb[2] : m;               tc[3] = g2 ? tc[2] : id;
                    tb[2] = g2 ? (g1 ? tb[1] : m) : tb[2]; tc[2] = g2 ? (g1 ? tc[1] : id) : tc[2];
                    tb[1] = g1 ? (g0 ? tb[0] : m) : tb[1]; tc[1] = g1 ? (g0 ? tc[0] : id) : tc[1];
                    tb[0] = g0 ? m : tb[0];               tc[0] = g0 ? id : tc[0];
                  } else {
                    // slot i takes the entry above it when m beats both, m when it beats slot i only (always true of the last)
                    bool gt[TOPC - 1];
#pragma unroll
                    for (int i = 0; i < TOPC - 1; ++i) gt[i] = m > tb[i];
                    tb[TOPC - 1] = gt[TOPC - 2] ? tb[TOPC - 2] : m; tc[TOPC - 1] = gt[TOPC - 2] ? tc[TOPC - 2] : id;
#pragma unroll
                    for (int i = TOPC - 2; i > 0; --i) {
                      tb[i] = gt[i] ? (gt[i - 1] ? tb[i - 1] : m) : tb[i];
                      tc[i] = gt[i] ? (gt[i - 1] ? tc[i - 1] : id) : tc[i];
                    }
                    tb[0] = gt[0] ? m : tb[0];               tc[0] = gt[0] ? id : tc[0];
                  }
                }
              }
            }
          }
          if (sd.block_max != nullptr) {   // warp-uniform: column side of mutual NN (hn_match_mutual)
            const long long rb = row >> 5;
            float* const bmax = BATCHED ? sd.block_max + static_cast<long long>(pair) * ((sd.Nb + kChunk - 1) / kChunk) * sd.n_row_blocks
                                        : nullptr;   // this pair's [ceil(Nb / 8)][n_row_blocks] slice
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
              const float half8[8] = {cm[hf * 8], cm[hf * 8 + 1], cm[hf * 8 + 2], cm[hf * 8 + 3],
                                      cm[hf * 8 + 4], cm[hf * 8 + 5], cm[hf * 8 + 6], cm[hf * 8 + 7]};
              const float bm = warp_chunk_max8(half8, lane);
              const long long cb = col0 / kChunk + hf * 8 + (lane >> 2);
              if ((lane & 3) == 0 && cb * kChunk < cols() && rb < sd.n_row_blocks) (BATCHED ? bmax : sd.block_max)[cb * sd.n_row_blocks + rb] = bm;
            }
          }
        } else {
          // NOT unrolled: the exact epilogue is ~80 instructions per column and a loss-sized problem (N = 1024) runs it ONCE per CTA,
          // so four unrolled copies were 10 k instructions of straight-line code fetched cold - the instruction fetch (stall reason
          // no_inst in ncu) was most of the kernel's 28 us; one copy of the 32-column body stays in the instruction cache.
#pragma unroll 1
          for (int c0 = CS == 1 ? 0 : cs * 32; c0 < (CS == 1 ? kDistTile : cs * 32 + 32); c0 += 32) {
            uint32_t r[32];
            tmem_ld32(t_row + c0, r);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const long long col = col0 + c0 + j;
              const float dot = __uint_as_float(r[j]) * p.dot_scale;
              float d;
              if (p.form == HN_FORM_HARDNET) {
                // sqrt((|a|^2 + |p|^2) - 2ab + 1e-6), hardnet/Losses.py:12-13
                const float s = (na + s_nb[acc * kDistTile + c0 + j]) - 2.0f * dot;
                d = sqrtf(s + 1e-6f);
              } else {
                // sqrt(clamp(2 - 2ab, 1e-8, 4)), FDLNet-master/utils/math_utils.py:15-18
                d = sqrtf(fminf(fmaxf(2.0f - 2.0f * dot, 1e-8f), 4.0f));
              }
              if (p.loss_mask) {
                d += 1e-8f;                                   // Losses.py:95
                if (col == row) {
                  if (sd.pos && row_ok) sd.pos[row] = d;      // Losses.py:99 (before masking)
                  d += 10.0f;                                 // Losses.py:100
                }
                if (d < 0.008f) d += 10.0f;                   // Losses.py:101-103
              }
              if (NEI) {
                if (col == row) {
                  if (sd.pos && row_ok) sd.pos[row] = d;      // rf_des.py:70 (before masking)
                  d += 10.0f;                                 // rf_des.py:71
                }
                // pairwise_distances(kp, kp).lt(C), math_utils.py:22-40: sqrt(clamp(|x|^2 + |y|^2 - 2 x.y, 1e-8)) < C
                const float4 cxy = s_xy[acc * kDistTile + c0 + j];
                const float da = (r_axy.x * r_axy.x + r_axy.y * r_axy.y) + (cxy.x * cxy.x + cxy.y * cxy.y) - 2.0f * (r_axy.x * cxy.x + r_axy.y * cxy.y);
                const float dp = (r_pxy.x * r_pxy.x + r_pxy.y * r_pxy.y) + (cxy.z * cxy.z + cxy.w * cxy.w) - 2.0f * (r_pxy.x * cxy.z + r_pxy.y * cxy.w);
                if (sqrtf(fmaxf(da, 1e-8f)) < p.nei_c) d += 10.0f;   // rf_des.py:74-79
                if (sqrtf(fmaxf(dp, 1e-8f)) < p.nei_c) d += 10.0f;   // rf_des.py:80-85
              }
              if (col < sd.Nb && d < best) { best = d; best_col = static_cast<int>(col); }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(acc));
      }

      if (row_ok) {
        if (EXACT) {
          if (sd.row_pack && best_col != 0x7fffffff) {
            const unsigned long long pk =
                (static_cast<unsigned long long>(__float_as_uint(best)) << 32) | static_cast<unsigned int>(best_col);
            atomicMin(sd.row_pack + row, pk);  // distances are positive: bit pattern is order preserving
          }
        } else {
          const long long out_row = BATCHED ? pair * sd.Na + row : row;   // chunk ids stay local to the pair
          store_cand_list(sd.cand, sd.cand_val, out_row * p.segments + seg, tb, tc);
          if constexpr (DROP) p.cand_drop[out_row * p.segments + seg] = drop;
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

}  // namespace hn
