// The opaque handle behind the C ABI: packed weights, static TMA descriptors and activation scratch.
#pragma once

#include <cuda_runtime.h>

#include <vector>

#include "../../include/hardnet_b200.h"
#include "tc_conv.cuh"

namespace hn {
// internal value of `in_dtype` next to HN_F32 / HN_U8: the input pointer is a HOST ClipSrc (clip.cuh) and the patches are cropped
// from the image stack by the front kernel's loader warps (hn_forward_clip)
constexpr int kInClip = 100;
struct NasState;
void nas_state_free(NasState* s);
// [rows, K] x [K, 128] + bias + L2 normalisation (hardnet_forward.cu); shared by the HardNet and NAS heads
int launch_head(const TcParams& p, int sm_count, cudaStream_t stream);
// input_norm (optional) + conv 1->32 k3 + BN + ReLU on the tensor core (hardnet_forward.cu); also the NAS stem
int launch_l1(const void* patches, int in_dtype, uint16_t* out, const float* w, const float* bias, float2* stats, int n,
              int act_bf16, int sm_count, cudaStream_t s, float norm_eps = 1e-7f);
// NAS front: stem + pointwise 32 -> 32 conv in one launch of the fused front kernel (hardnet_forward.cu)
int launch_front_pw(const void* patches, int in_dtype, uint16_t* out, const CUtensorMap& tm_out, const float* w1,
                    const float* bias1, const uint16_t* w2img, const float* bias2_host /*[32], HOST memory*/, int n, int act_bf16, int sm_count,
                    cudaStream_t s);
// the same with the stride-2 depthwise conv (fdw = 3 | 5) or max-pool (fdw = 1) behind it: output [n][16][16][32] NHWC fp16, or
// channel-planar [n][4][16][16][8] (out_planar: what the tail kernel bulk-copies)
int launch_front_pw_dw(const void* patches, int in_dtype, uint16_t* out, const float* w1, const float* bias1, const uint16_t* w2img,
                       const float* bias2_host, int fdw, const float* dw_w, const float* dw_b, int dw_relu, int n, int sm_count,
                       cudaStream_t s, int out_planar = 0);
void front_pw_weight_image(const uint16_t* w /*[32][32] 16-bit*/, std::vector<uint16_t>& img);
}  // namespace hn

// Run-time switches (A/B measurements, tests), read from the environment ONCE in hn_create: the hot calls never call getenv.
struct HnEnv {
  bool nas_front = true;      // HN_NAS_FRONT=0: stem and first pointwise conv as separate kernels
  bool nas_dw_smem = true;    // HN_NAS_DW_SMEM=0: register-strip depthwise / max-pool kernels
  bool nas_dw_sh8 = true;     // HN_NAS_DW_SH8=0: 4-row strips for every depthwise shape
  bool nas_front_dw = true;   // HN_NAS_FRONT_DW=0: the stride-2 depthwise conv / max-pool behind the stem as its own kernel
  bool nas_dw_f32 = false;    // HN_NAS_DW_F32=1: fp32 depthwise arithmetic also for fp16 activations (default: packed half2)
  bool nas_tail = true;       // HN_NAS_TAIL=0: no warpgroup-per-patch tail kernel (nas_tail.cuh) behind the fused front stage
  bool nas_fold = true;       // HN_NAS_FOLD=0: the tail runs the packed ops one by one (no folding of linear 1x1 convs into their consumers)
  int nas_tail_cut = 2;       // HN_NAS_TAIL_CUT: start a new tail launch at a block boundary whose tensor is <= 1/cut of the launch's
                              // input (smaller maps -> smaller buffers -> more warpgroups per SM); 0 = one launch for the whole tail
  int nas_tail_minops = 4;    // HN_NAS_TAIL_MINOPS: ... and only if at least this many ops remain behind the cut
  int nas_tail_wg = 6;        // HN_NAS_TAIL_WG: cap on warpgroups (patches in flight) per CTA
};

struct hn_handle {
  HnEnv env;
  int chunk = 0;            // patches per conv-stack pass
  long long head_rows = 0;  // capacity of the L6 output buffer (patches)
  int sm_count = 0;
  bool packed = false;
  int act_bf16 = 0;
  uint16_t* act[2] = {nullptr, nullptr};  // ping-pong activations, chunk * 32*32*32 elements each
  uint16_t* l6 = nullptr;                 // [head_rows, 8, 8, 128]
  uint16_t* wconv[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};  // [cout][9*cin]
  uint16_t* whead = nullptr;                                           // [128][8192]
  float* w1 = nullptr;                                                 // [9][32]
  uint16_t* w2img = nullptr;  // conv2 weights as the fused front kernel's shared-memory image (front_fused.cuh)
  float* bias = nullptr;                                               // 7 x 128
  float norm_eps = 1e-7f;       // added to the per-patch std in input_norm (hn_set_hardnet_eps)
  float bias2_host[32] = {0};   // conv2's folded BN shift on the host: passed to the fused front kernel by value
  float* head_partial = nullptr;  // split-K partial sums of the head GEMM at small batches ([#SM][128][128] fp32)
  float2* stats = nullptr;                                             // per-patch (mean, 1/std), chunk entries
  hn::TcParams conv_params[5];   // 3x3 layers on the CTA-pair kernel (tc_conv_pair.cuh); [0] unused (conv2 is in the front kernel)
  hn::TcParams head_params;
  bool fuse34 = true;            // conv3 + conv4 in one kernel (tc_conv34.cuh); HN_FUSE34=0: two kernels, the reference of the
                                 // fused one. The deeper layers then read / write the other ping-pong buffer (act_buf)
  hn::Conv34Params c34;
  // optional per-stage CUDA-event timing (stage 0 = L1, 1..5 = 3x3 convs, 6 = head)
  unsigned profile_mask = 0;
  std::vector<cudaEvent_t> ev[7];
  size_t ev_used[7] = {0, 0, 0, 0, 0, 0, 0};
  hn::NasState* nas = nullptr;  // NAS-derived descriptor net (nas.cu)
};
