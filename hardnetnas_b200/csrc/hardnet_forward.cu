// HardNet.forward (hardnet/HardNet.py:312-315) behind the C ABI: weight packing (BatchNorm fold),
// static TMA descriptors over handle-owned activation scratch, and the per-chunk launch sequence
//   fused front (input_norm + conv1 + conv2, front_fused.cuh) -> fused conv3 + conv4 (tc_conv34.cuh) -> conv5, conv6
//   (tcgen05 implicit GEMM over channel-planar activations, tc_conv_pair.cuh) -> head GEMM + L2Norm.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <vector>

#include "front_fused.cuh"
#include "handle.h"
#include "host_common.h"
#include "l1_tc.cuh"
#include "tc_conv.cuh"
#include "tc_conv_pair.cuh"
#include "tc_conv34.cuh"

namespace hn {

struct ConvLayer {
  int cin, cout, stride, hin, hout;
};
// features[3], [6], [9], [12], [15] of hardnet/HardNet.py:284-298
static const ConvLayer kConv[5] = {
    {32, 32, 1, 32, 32}, {32, 64, 2, 32, 16}, {64, 64, 1, 16, 16}, {64, 128, 2, 16, 8}, {128, 128, 1, 8, 8}};

constexpr int kHeadK = 8 * 8 * 128;

}  // namespace hn


namespace hn {

// Event pair around one launch of an instrumented stage (events are created on demand and reused).
struct StageTimer {
  hn_handle* h;
  int stage;
  cudaStream_t s;
  bool on;
  StageTimer(hn_handle* h_, int stage_, cudaStream_t s_) : h(h_), stage(stage_), s(s_), on((h_->profile_mask >> stage_) & 1u) {
    if (on) record();
  }
  ~StageTimer() {
    if (on) record();
  }
  void record() {
    auto& v = h->ev[stage];
    size_t& u = h->ev_used[stage];
    if (u == v.size()) {
      cudaEvent_t e;
      if (cudaEventCreate(&e) != cudaSuccess) { on = false; return; }
      v.push_back(e);
    }
    cudaEventRecord(v[u++], s);
  }
};

template <int CIN, int COUT, int HOUT, int STRIDE, int STAGES, bool ROWSHIFT, bool OUT_PARITY, int KCB_ = 0>
static int launch_conv_pair_cfg(const TcParams& p, int sm_count, cudaStream_t stream) {
  using C = PairCfg<CIN, COUT, HOUT, STRIDE, STAGES, ROWSHIFT, KCB_>;
  auto kern = conv3x3_pair_kernel<CIN, COUT, HOUT, STRIDE, STAGES, ROWSHIFT, OUT_PARITY, KCB_>;
  static DeviceOnce attr_once;  // per instantiation
  if (attr_once.first_time()) {
    HN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(C::SMEM)));
  }
  if (p.num_tiles <= 0) return HN_OK;
  const int groups = (p.num_tiles + 1) / 2;
  const int grid = 2 * std::min(groups, sm_count / 2);   // whole CTA pairs (__cluster_dims__(2, 1, 1))
  kern<<<grid, kTcThreads, C::SMEM, stream>>>(p);
  HN_CUDA(cudaGetLastError());
  count_launch();
  return HN_OK;
}

// conv2 (li = 0) lives in the fused front kernel. Every 3x3 layer runs on CTA pairs (cta_group::2): weights resident (half per
// CTA), M = 256 per MMA. OUT_PARITY: the consumer is a stride-2 conv and wants parity sub-planes.
static const bool kRowShift[5] = {false, false, true, false, true};
static const int kKcb[5] = {64, 64, 128, 128, 128};   // bytes of one pixel's channel chunk per k-block (PairCfg::KCB)

static int launch_conv(int li, const TcParams& p, int sm_count, cudaStream_t s) {
  switch (li) {   //                          CIN COUT HOUT STRIDE STAGES ROWSHIFT OUT_PARITY
    case 1: return launch_conv_pair_cfg<32, 64, 16, 2, 9, false, false>(p, sm_count, s);
    case 2: return launch_conv_pair_cfg<64, 64, 16, 1, 9, true, true>(p, sm_count, s);
    case 3: return launch_conv_pair_cfg<64, 128, 8, 2, 9, false, false>(p, sm_count, s);
    case 4: return launch_conv_pair_cfg<128, 128, 8, 1, 4, true, false>(p, sm_count, s);
  }
  return HN_ERR_INVALID;
}

// conv3 + conv4 in one kernel (tc_conv34.cuh): conv2 output in act[1] -> conv4 output in `out`.
static int launch_conv34(const Conv34Params& p, int sm_count, cudaStream_t stream) {
  static DeviceOnce attr_once;
  if (attr_once.first_time()) {
    HN_CUDA(cudaFuncSetAttribute(conv34_stack_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(C34SCfg::SMEM)));
  }
  if (p.n_patches <= 0) return HN_OK;
  const int groups = (p.n_patches + 1) / 2;
  const int grid = 2 * std::min(groups, sm_count / 2);   // whole CTA pairs (__cluster_dims__(2, 1, 1))
  conv34_stack_kernel<<<grid, kC34SThreads, C34SCfg::SMEM, stream>>>(p);
  HN_CUDA(cudaGetLastError());
  count_launch();
  return HN_OK;
}

static int build_conv34_params(hn_handle* h) {
  Conv34Params& p = h->c34;
  memset(&p, 0, sizeof(p));
  if (!h->fuse34) return HN_OK;
  const uint16_t* in = h->act[1];   // conv2 output: parity sub-planes [patch][4 planes][ypar][xpar][16][16][8]
  const uint32_t box[4] = {16 * 8, 9, 1, 4};
  for (int ypar = 0; ypar < 2; ++ypar)
    for (int xpar = 0; xpar < 2; ++xpar) {
      const uint64_t dims[4] = {16 * 8, 16, static_cast<uint64_t>(h->chunk), 4};
      const uint64_t str[3] = {16 * 16, 32ull * 32 * 32 * 2, 32 * 32 * 16};
      HN_TRY(make_tmap_16bit(&p.tmA[ypar * 2 + xpar], in + (ypar * 2 + xpar) * 16 * 16 * 8, 4, dims, str, box, 0));
    }
  {
    const uint64_t dims[2] = {9 * 32, 64};
    const uint64_t str[1] = {9 * 32 * 2};
    const uint32_t wbox[2] = {32, 32};
    HN_TRY(make_tmap_16bit(&p.tmB3, h->wconv[1], 2, dims, str, wbox, 64));
  }
  {
    const uint64_t dims[2] = {9 * 64, 64};
    const uint64_t str[1] = {9 * 64 * 2};
    const uint32_t wbox[2] = {64, 32};
    HN_TRY(make_tmap_16bit(&p.tmB4, h->wconv[2], 2, dims, str, wbox, 128));
  }
  return HN_OK;
}

static int run_conv34(hn_handle* h, int n, void* out, cudaStream_t s) {
  Conv34Params p = h->c34;
  p.n_patches = n;
  p.act_bf16 = h->act_bf16;
  p.out = out;
  StageTimer timer(h, 2, s);   // reported as the conv3 stage; the conv4 stage then has no launches of its own
  return launch_conv34(p, h->sm_count, s);
}

// Stage 1 (input_norm + conv 1->32 + BN + ReLU) on the tensor core; do_norm = 0 gives the NAS stem.
int launch_l1(const void* patches, int in_dtype, uint16_t* out, const float* w, const float* bias, float2* stats, int n,
              int act_bf16, int sm_count, cudaStream_t s, float norm_eps) {
  static DeviceOnce attr_once;
  if (attr_once.first_time()) {
    HN_CUDA(cudaFuncSetAttribute(l1_tc_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kL1TcSmem)));
    HN_CUDA(cudaFuncSetAttribute(l1_tc_kernel<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kL1TcSmem)));
  }
  if (n <= 0) return HN_OK;
  const int grid = std::min(n, sm_count);
  const int sgrid = std::min((n + 7) / 8, sm_count * 8);
  if (in_dtype == HN_F32) {
    const float* x = static_cast<const float*>(patches);
    if (stats) patch_stats_kernel<float><<<sgrid, 256, 0, s>>>(x, stats, n, norm_eps);
    l1_tc_kernel<float><<<grid, kL1TcThreads, kL1TcSmem, s>>>(x, out, w, bias, stats, n, act_bf16);
  } else {
    const uint8_t* x = static_cast<const uint8_t*>(patches);
    if (stats) patch_stats_kernel<uint8_t><<<sgrid, 256, 0, s>>>(x, stats, n, norm_eps);
    l1_tc_kernel<uint8_t><<<grid, kL1TcThreads, kL1TcSmem, s>>>(x, out, w, bias, stats, n, act_bf16);
  }
  HN_CUDA(cudaGetLastError());
  count_launch(stats ? 2 : 1);
  return HN_OK;
}

// Stage 1 + conv2 fused (front_fused.cuh): patches -> conv2 output (NHWC 16-bit), stage-1 activation stays on chip.
static int launch_front_fused(hn_handle* h, const void* patches, int in_dtype, uint16_t* out, int n, cudaStream_t s) {
  static DeviceOnce attr_once;
  if (attr_once.first_time()) {
    HN_CUDA(cudaFuncSetAttribute(front_fused_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kFfSmem)));
    HN_CUDA(cudaFuncSetAttribute(front_fused_kernel<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kFfSmem)));
  }
  if (n <= 0) return HN_OK;
  const int grid = std::min(n, h->sm_count);
  const uint4* w2 = reinterpret_cast<const uint4*>(h->w2img);
  static const CUtensorMap no_map = {};   // output tensor map: only the pointwise (NAS) variant stores through TMA
  FfBias b2;
  memcpy(b2.v, h->bias2_host, sizeof(b2.v));
  if (in_dtype == kInClip) {   // `patches` is a HOST ClipSrc: the loader warps crop the patches from the image stack
    static DeviceOnce clip_once;
    if (clip_once.first_time())
      HN_CUDA(cudaFuncSetAttribute(front_fused_clip_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kFfSmem)));
    front_fused_clip_kernel<<<grid, kFfThreads, kFfSmem, s>>>(*static_cast<const ClipSrc*>(patches), out, h->w1, h->bias, w2, b2, n,
                                                             h->act_bf16, h->norm_eps, no_map);
  } else if (in_dtype == HN_F32) {
    const float* x = static_cast<const float*>(patches);
    front_fused_kernel<float><<<grid, kFfThreads, kFfSmem, s>>>(x, out, h->w1, h->bias, w2, b2, 1, n, h->act_bf16, h->norm_eps, no_map);
  } else {
    const uint8_t* x = static_cast<const uint8_t*>(patches);
    front_fused_kernel<uint8_t><<<grid, kFfThreads, kFfSmem, s>>>(x, out, h->w1, h->bias, w2, b2, 1, n, h->act_bf16, h->norm_eps, no_map);
  }
  HN_CUDA(cudaGetLastError());
  count_launch(1);
  return HN_OK;
}

// NAS front: stem (1 -> 32, 3x3, folded BN, ReLU) + the first block's pointwise 32 -> 32 conv (folded BN, ReLU) in one
// launch of the fused front kernel (PW2 variant); `w2img` is a front-kernel weight image whose centre tap is the 1x1 conv.
int launch_front_pw(const void* patches, int in_dtype, uint16_t* out, const CUtensorMap& tm_out, const float* w1,
                    const float* bias1, const uint16_t* w2img, const float* bias2_host, int n, int act_bf16, int sm_count,
                    cudaStream_t s) {
  static DeviceOnce attr_once;
  if (attr_once.first_time()) {
    HN_CUDA(cudaFuncSetAttribute(front_fused_kernel<float, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kFfSmem)));
    HN_CUDA(cudaFuncSetAttribute(front_fused_kernel<uint8_t, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kFfSmem)));
  }
  if (n <= 0) return HN_OK;
  const int grid = std::min(n, sm_count);
  const uint4* w2 = reinterpret_cast<const uint4*>(w2img);
  FfBias bias2;
  memcpy(bias2.v, bias2_host, sizeof(bias2.v));
  if (in_dtype == HN_F32)
    front_fused_kernel<float, true><<<grid, kFfThreads, kFfSmem, s>>>(static_cast<const float*>(patches), out, w1, bias1, w2, bias2, 0, n, act_bf16, 0.f, tm_out);
  else
    front_fused_kernel<uint8_t, true><<<grid, kFfThreads, kFfSmem, s>>>(static_cast<const uint8_t*>(patches), out, w1, bias1, w2, bias2, 0, n, act_bf16, 0.f, tm_out);
  HN_CUDA(cudaGetLastError());
  count_launch(1);
  return HN_OK;
}

// NAS front with the block's stride-2 depthwise conv (fdw = 3 | 5) or max-pool (fdw = 1) fused behind the pointwise stage
// (FDW variant of the front kernel): patches -> [n][16][16][32] NHWC fp16; the 64 KB/patch pointwise output stays on chip.
int launch_front_pw_dw(const void* patches, int in_dtype, uint16_t* out, const float* w1, const float* bias1, const uint16_t* w2img,
                       const float* bias2_host, int fdw, const float* dw_w, const float* dw_b, int dw_relu, int n, int sm_count,
                       cudaStream_t s, int out_planar) {
  static DeviceOnce attr_once;
  if (attr_once.first_time()) {
#define HN_FDW_ATTR(T, F) HN_CUDA(cudaFuncSetAttribute(front_fused_kernel<T, true, F>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kFfSmem)))
    HN_FDW_ATTR(float, 1); HN_FDW_ATTR(float, 3); HN_FDW_ATTR(float, 5);
    HN_FDW_ATTR(uint8_t, 1); HN_FDW_ATTR(uint8_t, 3); HN_FDW_ATTR(uint8_t, 5);
#undef HN_FDW_ATTR
  }
  if (n <= 0) return HN_OK;
  const int grid = std::min(n, sm_count);
  const uint4* w2 = reinterpret_cast<const uint4*>(w2img);
  static const CUtensorMap no_map = {};
  FfBias bias2;
  memcpy(bias2.v, bias2_host, sizeof(bias2.v));
#define HN_FDW_LAUNCH(T, F) front_fused_kernel<T, true, F><<<grid, kFfThreads, kFfSmem, s>>>(static_cast<const T*>(patches), out, w1, bias1, w2, bias2, 0, n, 0, 0.f, no_map, dw_w, dw_b, dw_relu, out_planar)
  if (in_dtype == HN_F32) {
    if (fdw == 1) HN_FDW_LAUNCH(float, 1); else if (fdw == 3) HN_FDW_LAUNCH(float, 3); else HN_FDW_LAUNCH(float, 5);
  } else {
    if (fdw == 1) HN_FDW_LAUNCH(uint8_t, 1); else if (fdw == 3) HN_FDW_LAUNCH(uint8_t, 3); else HN_FDW_LAUNCH(uint8_t, 5);
  }
#undef HN_FDW_LAUNCH
  HN_CUDA(cudaGetLastError());
  count_launch(1);
  return HN_OK;
}

// Front-kernel weight image (front_fused.cuh) of a pointwise 32 -> 32 conv: [co][ci] 16-bit weights at the centre tap.
void front_pw_weight_image(const uint16_t* w /*[32][32]*/, std::vector<uint16_t>& img) {
  img.assign(kFfW2 / 2, 0);
  for (int co = 0; co < 32; ++co)
    for (int ci = 0; ci < 32; ++ci) {
      const int nn = 32 + co;
      const size_t byte = static_cast<size_t>(kFfW2Tap) + (nn >> 3) * 512 + (ci >> 3) * 128 + (nn & 7) * 16 + (ci & 7) * 2;
      img[byte / 2] = w[co * 32 + ci];
    }
}

int launch_head(const TcParams& p_in, int sm_count, cudaStream_t stream) {
  static DeviceOnce attr_once;
  if (attr_once.first_time()) {
    HN_CUDA(cudaFuncSetAttribute(gemm_l2norm_kernel<kHeadN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(kHeadSmem)));
    HN_CUDA(cudaFuncSetAttribute(gemm_l2norm_kernel<kHeadN, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(kHeadSmem)));
  }
  if (p_in.num_tiles <= 0) return HN_OK;
  TcParams p = p_in;
  // Small batches: a 128-row tile streams the whole K x 128 weight matrix (2 MB for HardNet's 8 x 8 head) through ONE SM, so a
  // 1024-patch head took 41 us on 8 CTAs against 4 us at the bulk rate. Split K over up to 16 CTAs per tile (raw fp32
  // partials, summed with the bias and normalised by head_finalize_kernel) whenever the tiles alone fill less than half of the
  // machine. (Changes the last bit of a descriptor relative to the unsplit head: a different fp32 summation order.)
  int splits = 1;
  if (p.partial != nullptr && p.num_tiles * 2 <= sm_count) {
    while (splits * 2 <= 16 && p.num_tiles * splits * 2 <= sm_count && p.num_k_stages % (splits * 2) == 0) splits *= 2;
  }
  p.k_splits = splits;
  const int items = p.num_tiles * splits;
  if (splits == 1 && p.num_tiles > sm_count) {
    // bulk batches: two row tiles per streamed weight block (the kernel is bound by the L2 -> SM traffic)
    gemm_l2norm_kernel<kHeadN, 2><<<std::min((p.num_tiles + 1) / 2, sm_count), kTcThreads, kHeadSmem, stream>>>(p);
    HN_CUDA(cudaGetLastError());
    count_launch();
    return HN_OK;
  }
  gemm_l2norm_kernel<kHeadN><<<std::min(items, sm_count), kTcThreads, kHeadSmem, stream>>>(p);
  HN_CUDA(cudaGetLastError());
  count_launch();
  if (splits > 1) {
    const int threads = 256;
    head_finalize_kernel<<<static_cast<unsigned>((p.total_rows * 32 + threads - 1) / threads), threads, 0, stream>>>(
        p.partial, splits, static_cast<long long>(p.num_tiles) * kTileM, p.total_rows, p.bias, p.l2_eps, p.out, p.out_dtype);
    HN_CUDA(cudaGetLastError());
    count_launch();
  }
  return HN_OK;
}

static uint16_t to16(float v, int bf16) {
  if (bf16) {
    __nv_bfloat16 h = __float2bfloat16_rn(v);
    return *reinterpret_cast<uint16_t*>(&h);
  }
  __half h = __float2half_rn(v);
  return *reinterpret_cast<uint16_t*>(&h);
}

// The ping-pong buffer that holds the output of `stage` (1 = stage 1, 2 = conv2 ... 5 = conv5; conv6 writes l6). The front
// kernel writes act[1] and the stages alternate. With conv3 + conv4 fused the conv4 output lands in act[0] (the fused kernel
// cannot write the buffer it reads), so conv4 and conv5 use the opposite buffers.
static uint16_t* act_buf(const hn_handle* h, int stage) {
  return h->act[((stage - 1) & 1) ^ ((h->fuse34 && stage >= 4) ? 1 : 0)];
}

// Static descriptors of one 3x3 layer over the handle's buffers; only the tile counts change per call.
// kcb = bytes of one pixel's channel chunk per k-block; the weight box covers the C_out / 2 rows of one CTA of the pair.
static int build_conv_params(hn_handle* h, int li, int kcb, bool rowshift, TcParams& p) {
  const ConvLayer& L = kConv[li];
  memset(&p, 0, sizeof(p));
  const int kc = kcb / 2;
  const uint16_t* in = act_buf(h, li + 1);   // the output of the layer before (stage li + 1)
  const int pix_out = L.hout * L.hout;
  const int rows_per_tile = pix_out >= kTileM ? kTileM / L.hout : L.hout;
  const int patches_per_tile = pix_out >= kTileM ? 1 : kTileM / pix_out;
  // channel-planar input [patch][plane][y][x][8] seen as (x * 8, y, patch, plane); box = whole rows of NPL planes.
  // ROWSHIFT layers order the box (x * 8, patch, y, plane) instead (see PairCfg).
  const uint64_t C = L.cin, W = L.hin, H = L.hin;
  if (L.stride == 1 && rowshift) {
    const uint32_t box[4] = {static_cast<uint32_t>(L.hout * 8), static_cast<uint32_t>(patches_per_tile),
                             static_cast<uint32_t>(rows_per_tile + 2), static_cast<uint32_t>(kc / 8)};
    const uint64_t dims[4] = {W * 8, static_cast<uint64_t>(h->chunk), H, C / 8};
    const uint64_t str[3] = {C * H * W * 2, W * 16, H * W * 16};
    HN_TRY(make_tmap_16bit(&p.tmA[0], in, 4, dims, str, box, 0));
  } else if (L.stride == 1) {
    const uint32_t box[4] = {static_cast<uint32_t>(L.hout * 8), static_cast<uint32_t>(rows_per_tile),
                             static_cast<uint32_t>(patches_per_tile), static_cast<uint32_t>(kc / 8)};
    const uint64_t dims[4] = {W * 8, H, static_cast<uint64_t>(h->chunk), C / 8};
    const uint64_t str[3] = {W * 16, C * H * W * 2, H * W * 16};
    HN_TRY(make_tmap_16bit(&p.tmA[0], in, 4, dims, str, box, 0));
  } else {
    // parity sub-planes [patch][plane][ypar][xpar][y/2][x/2][8]
    const uint32_t box[4] = {static_cast<uint32_t>(L.hout * 8), static_cast<uint32_t>(rows_per_tile),
                             static_cast<uint32_t>(patches_per_tile), static_cast<uint32_t>(kc / 8)};
    for (int ypar = 0; ypar < 2; ++ypar)
      for (int xpar = 0; xpar < 2; ++xpar) {
        const uint64_t dims[4] = {W / 2 * 8, H / 2, static_cast<uint64_t>(h->chunk), C / 8};
        const uint64_t str[3] = {W / 2 * 16, C * H * W * 2, H * W * 16};
        const uint16_t* base = in + (ypar * 2 + xpar) * (H / 2) * (W / 2) * 8;
        HN_TRY(make_tmap_16bit(&p.tmA[ypar * 2 + xpar], base, 4, dims, str, box, 0));
      }
  }
  {
    const uint64_t K = 9ull * L.cin;
    const uint64_t dims[2] = {K, static_cast<uint64_t>(L.cout)};
    const uint64_t str[1] = {K * 2};
    const uint32_t wbox[2] = {static_cast<uint32_t>(kc), static_cast<uint32_t>(L.cout / 2)};
    HN_TRY(make_tmap_16bit(&p.tmB, h->wconv[li], 2, dims, str, wbox, kcb));
  }
  p.bias = h->bias + 128 * (li + 1);
  return HN_OK;
}

static int build_params(hn_handle* h) {
  for (int li = 1; li < 5; ++li) {   // conv2 (li = 0) is part of the fused front kernel
    HN_TRY(build_conv_params(h, li, kKcb[li], kRowShift[li], h->conv_params[li]));
  }
  {
    TcParams& p = h->head_params;
    memset(&p, 0, sizeof(p));
    const uint64_t dimsA[2] = {kHeadK, static_cast<uint64_t>(h->head_rows)};
    const uint64_t strA[1] = {kHeadK * 2ull};
    const uint32_t boxA[2] = {64, kTileM};
    HN_TRY(make_tmap_16bit(&p.tmA[0], h->l6, 2, dimsA, strA, boxA, 128));
    const uint64_t dimsB[2] = {kHeadK, 128};
    const uint32_t boxB[2] = {64, 128};
    HN_TRY(make_tmap_16bit(&p.tmB, h->whead, 2, dimsB, strA, boxB, 128));
    p.num_k_stages = kHeadK / (64 * kHeadG);
    p.bias = h->bias + 128 * 6;
    p.l2_eps = 1e-10f;
  }
  HN_TRY(build_conv34_params(h));
  return HN_OK;
}

static int run_one_conv(hn_handle* h, int li, int n, void* out, cudaStream_t s) {
  const ConvLayer& L = kConv[li];
  TcParams p = h->conv_params[li];
  const long long pix_out = static_cast<long long>(L.hout) * L.hout;
  p.total_rows = pix_out * n;
  p.num_tiles = static_cast<int>((p.total_rows + kTileM - 1) / kTileM);
  p.act_bf16 = h->act_bf16;
  p.out = out;
  StageTimer timer(h, li + 1, s);
  return launch_conv(li, p, h->sm_count, s);
}

// The input `off` patches further on: a pointer into the patch tensor, or (kInClip) a copy of the host ClipSrc whose first
// keypoint is moved on.
static const void* input_at(const void* patches, int in_dtype, long long off, ClipSrc* tmp) {
  if (in_dtype == kInClip) {
    *tmp = *static_cast<const ClipSrc*>(patches);
    tmp->n0 += off;
    return tmp;
  }
  return static_cast<const char*>(patches) + static_cast<size_t>(off) * 1024 * (in_dtype == HN_F32 ? 4 : 1);
}

// Runs the conv stack up to `last_layer` for `n` patches (n <= chunk); the conv6 output lands in l6 + l6_row * 8192.
static int run_conv_stack(hn_handle* h, const void* patches, int in_dtype, int n, long long l6_row, int last_layer,
                          cudaStream_t s) {
  if (last_layer < 2) {
    if (in_dtype == kInClip) {
      set_error("the stage-1 activation dump takes a patch tensor (crop with hn_clip_patches first)");
      return HN_ERR_INVALID;
    }
    StageTimer timer(h, 0, s);  // stage 1 alone (activation dump only), NHWC
    return launch_l1(patches, in_dtype, act_buf(h, 1), h->w1, h->bias, h->stats, n, h->act_bf16, h->sm_count, s, h->norm_eps);
  }
  {
    StageTimer timer(h, 1, s);  // stage 1 + conv2 (the stage-1 activation never reaches global memory)
    HN_TRY(launch_front_fused(h, patches, in_dtype, act_buf(h, 2), n, s));
  }
  const bool fuse = h->fuse34 && last_layer >= 4;   // a dump of conv3's own output runs the layer on its own
  if (fuse) HN_TRY(run_conv34(h, n, act_buf(h, 4), s));
  else if (last_layer >= 3) HN_TRY(run_one_conv(h, 1, n, act_buf(h, 3), s));
  for (int li = fuse ? 3 : 2; li < 5 && li + 2 <= last_layer; ++li)
    HN_TRY(run_one_conv(h, li, n, (li == 4) ? static_cast<void*>(h->l6 + l6_row * kHeadK) : static_cast<void*>(act_buf(h, li + 2)), s));
  return HN_OK;
}

}  // namespace hn

using namespace hn;

extern "C" int hn_create(hn_handle** out, int chunk_patches, long long head_rows) {
  HN_REQUIRE(out != nullptr, "hn_create: out is NULL");
  *out = nullptr;
  int dev = 0, major = 0;
  HN_CUDA(cudaGetDevice(&dev));
  HN_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) {
    set_error("hn_create: device compute capability %d.x is not sm_100 (no fallback path exists)", major);
    return HN_ERR_UNSUPPORTED;
  }
  hn_handle* h = new hn_handle();
  int st = device_sm_count(&h->sm_count);
  if (st != HN_OK) { delete h; return st; }
  if (chunk_patches <= 0) chunk_patches = h->sm_count * 128;  // measured: larger passes amortise launch + prologue cost
  chunk_patches = (chunk_patches + 1) & ~1;
  if (head_rows <= 0) head_rows = 2ll * h->sm_count * kTileM;   // two row tiles per CTA and head launch (gemm_l2norm_kernel<N, 2>)
  head_rows = std::max<long long>(head_rows, chunk_patches);
  head_rows = (head_rows + chunk_patches - 1) / chunk_patches * chunk_patches;
  h->chunk = chunk_patches;
  h->head_rows = head_rows;
  {
    auto flag = [](const char* name, bool dflt) { const char* e = getenv(name); return e ? e[0] != '0' : dflt; };
    auto num = [](const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; };
    h->env.nas_front = flag("HN_NAS_FRONT", true);
    h->env.nas_dw_smem = flag("HN_NAS_DW_SMEM", true);
    h->env.nas_dw_sh8 = flag("HN_NAS_DW_SH8", true);
    h->env.nas_dw_f32 = flag("HN_NAS_DW_F32", false);
    h->env.nas_front_dw = flag("HN_NAS_FRONT_DW", true);
    h->env.nas_tail = flag("HN_NAS_TAIL", true);
    h->env.nas_fold = flag("HN_NAS_FOLD", true);
    h->env.nas_tail_cut = std::max(0, num("HN_NAS_TAIL_CUT", 2));
    h->env.nas_tail_minops = std::max(1, num("HN_NAS_TAIL_MINOPS", 4));
    h->env.nas_tail_wg = std::min(6, std::max(1, num("HN_NAS_TAIL_WG", 6)));
    // HN_FUSE34=0: conv3 and conv4 as two kernels (the reference the fused kernel is tested against)
    h->fuse34 = flag("HN_FUSE34", true);
  }
  const size_t act_elems = static_cast<size_t>(chunk_patches) * 32 * 32 * 32;
  auto fail = [&](int code) { hn_destroy(h); return code; };
#define HN_CUDA_H(expr)                                                                                     \
  do {                                                                                                      \
    cudaError_t e__ = (expr);                                                                               \
    if (e__ != cudaSuccess) {                                                                               \
      set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__));                      \
      return fail(HN_ERR_CUDA);                                                                             \
    }                                                                                                       \
  } while (0)
  HN_CUDA_H(cudaMalloc(&h->act[0], act_elems * 2));
  HN_CUDA_H(cudaMalloc(&h->act[1], act_elems * 2));
  HN_CUDA_H(cudaMalloc(&h->l6, static_cast<size_t>(head_rows) * kHeadK * 2));
  // zero once so that never-written tail rows read as finite values
  HN_CUDA_H(cudaMemset(h->act[0], 0, act_elems * 2));
  HN_CUDA_H(cudaMemset(h->act[1], 0, act_elems * 2));
  HN_CUDA_H(cudaMemset(h->l6, 0, static_cast<size_t>(head_rows) * kHeadK * 2));
  for (int li = 0; li < 5; ++li)
    HN_CUDA_H(cudaMalloc(&h->wconv[li], static_cast<size_t>(kConv[li].cout) * 9 * kConv[li].cin * 2));
  HN_CUDA_H(cudaMalloc(&h->whead, static_cast<size_t>(128) * kHeadK * 2));
  HN_CUDA_H(cudaMalloc(&h->w1, 9 * 32 * sizeof(float)));
  HN_CUDA_H(cudaMalloc(&h->w2img, kFfW2));
  HN_CUDA_H(cudaMalloc(&h->bias, 7 * 128 * sizeof(float)));
  HN_CUDA_H(cudaMalloc(&h->stats, static_cast<size_t>(chunk_patches) * sizeof(float2)));
  // split-K partials of the head at small batches: tiles x splits <= #SM work items of 128 x 128 fp32 each
  HN_CUDA_H(cudaMalloc(&h->head_partial, static_cast<size_t>(h->sm_count) * kTileM * kHeadN * sizeof(float)));
#undef HN_CUDA_H
  st = build_params(h);
  if (st != HN_OK) return fail(st);
  *out = h;
  return HN_OK;
}

extern "C" int hn_destroy(hn_handle* h) {
  if (!h) return HN_OK;
  cudaFree(h->act[0]);
  cudaFree(h->act[1]);
  cudaFree(h->l6);
  for (int li = 0; li < 5; ++li) cudaFree(h->wconv[li]);
  cudaFree(h->whead);
  cudaFree(h->w1);
  cudaFree(h->w2img);
  cudaFree(h->bias);
  cudaFree(h->stats);
  cudaFree(h->head_partial);
  for (auto& v : h->ev)
    for (cudaEvent_t e : v) cudaEventDestroy(e);
  nas_state_free(h->nas);
  delete h;
  return HN_OK;
}

extern "C" int hn_set_hardnet_eps(hn_handle* h, float input_norm_eps, float l2_eps) {
  HN_REQUIRE(h, "hn_set_hardnet_eps: NULL handle");
  HN_REQUIRE(input_norm_eps >= 0.f && l2_eps >= 0.f, "hn_set_hardnet_eps: negative epsilon");
  h->norm_eps = input_norm_eps;
  h->head_params.l2_eps = l2_eps;
  return HN_OK;
}

extern "C" int hn_pack_hardnet(hn_handle* h, const float* const w[7], const float* const bn_mean[7],
                               const float* const bn_var[7], float bn_eps, int act_dtype) {
  HN_REQUIRE(h && w && bn_mean && bn_var, "hn_pack_hardnet: NULL argument");
  HN_REQUIRE(act_dtype == HN_F16 || act_dtype == HN_BF16, "hn_pack_hardnet: act_dtype must be HN_F16 or HN_BF16");
  for (int i = 0; i < 7; ++i) HN_REQUIRE(w[i] && bn_mean[i] && bn_var[i], "hn_pack_hardnet: NULL tensor %d", i);
  const int bf = act_dtype == HN_BF16;
  // Packing is rare and synchronous: forwards still queued on any stream (PyTorch's side streams are non-blocking, i.e. not
  // ordered against the legacy stream these copies use) must finish reading the old weights first ...
  HN_CUDA(cudaDeviceSynchronize());
  static const int cout[7] = {32, 32, 64, 64, 128, 128, 128};
  std::vector<float> bias(7 * 128, 0.f);
  std::vector<float> scale(128);
  // stage 1: [co][1][3][3] -> [tap][co] fp32
  {
    std::vector<float> w1(9 * 32);
    for (int co = 0; co < 32; ++co) {
      const float s = 1.0f / std::sqrt(bn_var[0][co] + bn_eps);
      bias[co] = -bn_mean[0][co] * s;
      for (int tap = 0; tap < 9; ++tap) w1[tap * 32 + co] = w[0][co * 9 + tap] * s;
    }
    HN_CUDA(cudaMemcpy(h->w1, w1.data(), w1.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  // 3x3 stages: OIHW -> [co][(ky*3+kx)*cin + ci], BN scale folded, 16-bit
  for (int li = 0; li < 5; ++li) {
    const ConvLayer& L = kConv[li];
    const int K = 9 * L.cin;
    std::vector<uint16_t> wp(static_cast<size_t>(L.cout) * K);
    for (int co = 0; co < L.cout; ++co) {
      const float s = 1.0f / std::sqrt(bn_var[li + 1][co] + bn_eps);
      bias[128 * (li + 1) + co] = -bn_mean[li + 1][co] * s;
      for (int ci = 0; ci < L.cin; ++ci)
        for (int tap = 0; tap < 9; ++tap)
          wp[static_cast<size_t>(co) * K + tap * L.cin + ci] = to16(w[li + 1][(static_cast<size_t>(co) * L.cin + ci) * 9 + tap] * s, bf);
    }
    HN_CUDA(cudaMemcpy(h->wconv[li], wp.data(), wp.size() * 2, cudaMemcpyHostToDevice));
    if (li == 0) {
      // fused front kernel: per ky a [n = kx * 32 + co][k = ci] tile in the UMMA no-swizzle K-major core-matrix order
      std::vector<uint16_t> img(kFfW2 / 2);
      for (int ky = 0; ky < 3; ++ky)
        for (int kx = 0; kx < 3; ++kx)
          for (int co = 0; co < 32; ++co)
            for (int ci = 0; ci < 32; ++ci) {
              const int nn = kx * 32 + co;
              const size_t byte = static_cast<size_t>(ky) * kFfW2Tap + (nn >> 3) * 512 + (ci >> 3) * 128 + (nn & 7) * 16 + (ci & 7) * 2;
              img[byte / 2] = wp[static_cast<size_t>(co) * K + (ky * 3 + kx) * 32 + ci];
            }
      HN_CUDA(cudaMemcpy(h->w2img, img.data(), img.size() * 2, cudaMemcpyHostToDevice));
    }
  }
  // head: [co][ci][8][8] -> [co][(ci/8)*512 + (y*8+x)*8 + ci%8]  (K order of the channel-planar conv6 output)
  {
    std::vector<uint16_t> wp(static_cast<size_t>(128) * kHeadK);
    for (int co = 0; co < 128; ++co) {
      const float s = 1.0f / std::sqrt(bn_var[6][co] + bn_eps);
      bias[128 * 6 + co] = -bn_mean[6][co] * s;
      for (int ci = 0; ci < 128; ++ci)
        for (int yx = 0; yx < 64; ++yx)
          wp[static_cast<size_t>(co) * kHeadK + (ci >> 3) * 512 + yx * 8 + (ci & 7)] = to16(w[6][(static_cast<size_t>(co) * 128 + ci) * 64 + yx] * s, bf);
    }
    HN_CUDA(cudaMemcpy(h->whead, wp.data(), wp.size() * 2, cudaMemcpyHostToDevice));
  }
  (void)cout;
  HN_CUDA(cudaMemcpy(h->bias, bias.data(), bias.size() * sizeof(float), cudaMemcpyHostToDevice));
  memcpy(h->bias2_host, bias.data() + 128, sizeof(h->bias2_host));
  memcpy(h->c34.bias3, bias.data() + 128 * 2, sizeof(h->c34.bias3));
  memcpy(h->c34.bias4, bias.data() + 128 * 3, sizeof(h->c34.bias4));
  for (int li = 0; li < 5; ++li)   // by-value copies for the conv kernels' epilogues
    memcpy(h->conv_params[li].bias_v, bias.data() + 128 * (li + 1), sizeof(h->conv_params[li].bias_v));
  // ... and every copy (small pageable H2D copies return once staged, before their DMA lands) must be complete before a
  // forward on another stream can read the new weights.
  HN_CUDA(cudaDeviceSynchronize());
  h->act_bf16 = bf;
  h->packed = true;
  return HN_OK;
}

static int forward_passes(hn_handle* h, const void* patches, int in_dtype, long long B, void* desc_out, int out_dtype, cudaStream_t s);

extern "C" int hn_forward(hn_handle* h, const void* patches, int in_dtype, long long B, void* desc_out, int out_dtype,
                          void* stream) {
  HN_REQUIRE(h, "hn_forward: NULL handle");
  if (!h->packed) {
    set_error("hn_forward: weights not packed (call hn_pack_hardnet first)");
    return HN_ERR_STATE;
  }
  HN_REQUIRE(B >= 0, "hn_forward: negative batch");
  HN_REQUIRE(in_dtype == HN_F32 || in_dtype == HN_U8, "hn_forward: in_dtype must be HN_F32 or HN_U8");
  HN_REQUIRE(out_dtype == HN_F32 || out_dtype == HN_F16 || out_dtype == HN_BF16 || out_dtype == HN_F8E4M3, "hn_forward: bad out_dtype");
  if (B == 0) return HN_OK;
  HN_REQUIRE(patches && desc_out, "hn_forward: NULL data pointer");
  return forward_passes(h, patches, in_dtype, B, desc_out, out_dtype, static_cast<cudaStream_t>(stream));
}

// Descriptors of patches that are cropped from the images on the fly: hn_clip_patches + hn_forward without the fp32 patch tensor
// (SURVEY.md section 8f row 2; reference caller FDLNet-master/.../rf_net_so.py:160-180 -> image_utils.py:11-158 -> des()).
extern "C" int hn_forward_clip(hn_handle* h, const void* images, int img_dtype, long long B, int H, int W, const long long* kpts_byxc,
                               const float* kpts_scale, const float* kpts_ori, const float* im_info, long long N, void* desc_out,
                               int out_dtype, void* stream) {
  HN_REQUIRE(h, "hn_forward_clip: NULL handle");
  if (!h->packed) {
    set_error("hn_forward_clip: weights not packed (call hn_pack_hardnet first)");
    return HN_ERR_STATE;
  }
  HN_REQUIRE(img_dtype == HN_F32 || img_dtype == HN_U8, "hn_forward_clip: img_dtype must be HN_F32 or HN_U8");
  HN_REQUIRE(out_dtype == HN_F32 || out_dtype == HN_F16 || out_dtype == HN_BF16 || out_dtype == HN_F8E4M3, "hn_forward_clip: bad out_dtype");
  HN_REQUIRE(B >= 1 && H >= 1 && W >= 1 && static_cast<long long>(H) * W < (1ll << 31), "hn_forward_clip: bad image size");
  HN_REQUIRE(N >= 0 && N % B == 0, "hn_forward_clip: the reference's view(B, -1) needs N (%lld) to be a multiple of B (%lld)", N, B);
  if (N == 0) return HN_OK;
  HN_REQUIRE(images && kpts_byxc && kpts_scale && im_info && desc_out, "hn_forward_clip: NULL argument");
  ClipSrc c;
  c.images = images;
  c.kpts_byxc = kpts_byxc;
  c.kpts_scale = kpts_scale;
  c.kpts_ori = kpts_ori;
  c.im_info = im_info;
  c.B = B;
  c.kp_per_image = N / B;
  c.n0 = 0;
  c.H = H;
  c.W = W;
  c.img_u8 = img_dtype == HN_U8;
  return forward_passes(h, &c, kInClip, N, desc_out, out_dtype, static_cast<cudaStream_t>(stream));
}

static int forward_passes(hn_handle* h, const void* patches, int in_dtype, long long B, void* desc_out, int out_dtype, cudaStream_t s) {
  const size_t out_elem = out_dtype == HN_F32 ? 4 : out_dtype == HN_F8E4M3 ? 1 : 2;
  for (long long base = 0; base < B; base += h->head_rows) {
    const long long nb = std::min<long long>(h->head_rows, B - base);
    for (long long off = 0; off < nb; off += h->chunk) {
      const int n = static_cast<int>(std::min<long long>(h->chunk, nb - off));
      ClipSrc clip_at;
      HN_TRY(run_conv_stack(h, input_at(patches, in_dtype, base + off, &clip_at), in_dtype, n, off, 6, s));
    }
    TcParams p = h->head_params;
    p.total_rows = nb;
    p.num_tiles = static_cast<int>((nb + kTileM - 1) / kTileM);
    p.act_bf16 = h->act_bf16;
    p.out_dtype = out_dtype;
    p.out = static_cast<char*>(desc_out) + static_cast<size_t>(base) * 128 * out_elem;
    p.partial = h->head_partial;
    StageTimer timer(h, 6, s);
    HN_TRY(launch_head(p, h->sm_count, s));
  }
  return HN_OK;
}

extern "C" int hn_forward_dump(hn_handle* h, const void* patches, int in_dtype, long long B, int layer, void* act_out,
                               void* stream) {
  HN_REQUIRE(h && patches && act_out, "hn_forward_dump: NULL argument");
  if (!h->packed) {
    set_error("hn_forward_dump: weights not packed");
    return HN_ERR_STATE;
  }
  HN_REQUIRE(layer >= 1 && layer <= 6, "hn_forward_dump: layer must be 1..6");
  HN_REQUIRE(B >= 1 && B <= h->chunk, "hn_forward_dump: B must be in [1, chunk=%d]", h->chunk);
  HN_REQUIRE(in_dtype == HN_F32 || in_dtype == HN_U8, "hn_forward_dump: bad in_dtype");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  HN_TRY(run_conv_stack(h, patches, in_dtype, static_cast<int>(B), 0, layer, s));
  static const size_t per_patch[7] = {0, 32 * 32 * 32, 32 * 32 * 32, 16 * 16 * 64, 16 * 16 * 64, 8 * 8 * 128, 8 * 8 * 128};
  const uint16_t* src = layer == 6 ? h->l6 : act_buf(h, layer);
  HN_CUDA(cudaMemcpyAsync(act_out, src, per_patch[layer] * 2 * static_cast<size_t>(B), cudaMemcpyDeviceToDevice, s));
  return HN_OK;
}

extern "C" int hn_profile_enable(hn_handle* h, unsigned stage_mask) {
  HN_REQUIRE(h, "hn_profile_enable: NULL handle");
  h->profile_mask = stage_mask & 0x7fu;
  for (size_t& u : h->ev_used) u = 0;
  return HN_OK;
}

extern "C" int hn_profile_read(hn_handle* h, double ms_out[7], long long launches_out[7]) {
  HN_REQUIRE(h && ms_out && launches_out, "hn_profile_read: NULL argument");
  for (int st = 0; st < 7; ++st) {
    double total = 0.0;
    const size_t pairs = h->ev_used[st] / 2;
    for (size_t i = 0; i < pairs; ++i) {
      HN_CUDA(cudaEventSynchronize(h->ev[st][2 * i + 1]));
      float ms = 0.f;
      HN_CUDA(cudaEventElapsedTime(&ms, h->ev[st][2 * i], h->ev[st][2 * i + 1]));
      total += ms;
    }
    ms_out[st] = total;
    launches_out[st] = static_cast<long long>(pairs);
    h->ev_used[st] = 0;
  }
  return HN_OK;
}

#ifdef HN_C34_TRACE
extern "C" int hn_debug_c34_trace(unsigned long long* out16, int reset) {
  HN_CUDA(cudaDeviceSynchronize());
  HN_CUDA(cudaMemcpyFromSymbol(out16, hn::hn_c34_trace, 16 * sizeof(unsigned long long)));
  if (reset) {
    unsigned long long z[16] = {0};
    HN_CUDA(cudaMemcpyToSymbol(hn::hn_c34_trace, z, sizeof(z)));
  }
  return HN_OK;
}
#endif

#ifdef HN_FF_TRACE
extern "C" int hn_debug_ff_trace(unsigned long long* out32, int reset) {
  HN_CUDA(cudaDeviceSynchronize());
  HN_CUDA(cudaMemcpyFromSymbol(out32, hn::hn_ff_trace, 32 * sizeof(unsigned long long)));
  if (reset) {
    unsigned long long z[32] = {0};
    HN_CUDA(cudaMemcpyToSymbol(hn::hn_ff_trace, z, sizeof(z)));
  }
  return HN_OK;
}
#endif
