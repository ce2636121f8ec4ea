/* hardnet_b200 — C ABI of the B200-native HardNet hot path.
 *
 * The reference (iamwangyabin/hardnetNas) is pure Python/PyTorch and has no FFI layer; its boundary is
 * the Python surface listed below. Each entry point here replaces the torch-op sequence behind one of
 * those Python symbols, and the Python mirror in hardnetnas_b200/ binds them with ctypes (the stub a
 * reference maintainer would add is shown in INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success or a negative hn_status; it never throws and never exits;
 *     hn_last_error() returns a thread-local, human readable description of the last failure.
 *   - data pointers are DEVICE pointers to contiguous buffers on the current CUDA device unless a
 *     parameter is documented as host memory; the caller owns every data buffer.
 *   - the library owns only what hangs off an hn_handle (packed weights, TMA descriptors, activation
 *     scratch). Handles are not thread safe; distinct handles are independent.
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no device-wide synchronisation
 *     and no allocation happens on the hot calls (hn_forward / hn_dist_min / hn_loss_hardnet / hn_match).
 *   - there is no CPU fallback: without a usable sm_100 device the calls fail with HN_ERR_CUDA.
 */
#ifndef HARDNET_B200_H_
#define HARDNET_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hn_handle hn_handle;

typedef enum hn_status {
  HN_OK = 0,
  HN_ERR_INVALID = -1,     /* bad argument (the reference's `assert` sites map here) */
  HN_ERR_CUDA = -2,        /* CUDA runtime / driver failure, see hn_last_error() */
  HN_ERR_STATE = -3,       /* e.g. forward before pack */
  HN_ERR_UNSUPPORTED = -4
} hn_status;

/* HN_F8E4M3: fp8 E4M3 (torch.float8_e4m3fn), descriptor outputs and matching rows only. 4 is not a dtype. */
typedef enum hn_dtype { HN_F32 = 0, HN_F16 = 1, HN_BF16 = 2, HN_U8 = 3, HN_F8E4M3 = 5 } hn_dtype;

/* distance forms */
#define HN_FORM_HARDNET 0 /* sqrt(|a|^2 + |p|^2 - 2ab + 1e-6)           hardnet/Losses.py:5-13            */
#define HN_FORM_FDL 1     /* sqrt(clamp(2 - 2ab, 1e-8, 4))              FDLNet-master/utils/math_utils.py:8-19 */

/* hn_dist_min flags */
#define HN_FLAG_LOSS_MASK 1 /* +1e-8, diagonal +10, (<0.008) +10        hardnet/Losses.py:95-103          */
#define HN_FLAG_SWAP 2      /* also produce column minima (anchor swap) hardnet/Losses.py:106-108         */
#define HN_FLAG_NEI_MASK 4  /* diagonal +10 and +10 per keypoint set whose two keypoints lie closer than C pixels
                               (HardNetNeiMask.loss, FDLNet-master/latency/rfnet/model/rf_des.py:66-86)      */

int hn_version(void);
const char* hn_last_error(void);
/* Kernels launched by this library since load (bench.py reports the delta over its timed region). */
long long hn_launch_count(void);

/* ---- handle -------------------------------------------------------------------------------------- */
/* chunk_patches: patches pushed through the conv stack per pass (0 = default, rounded to a multiple of
 * 2); head_rows: descriptors accumulated before the 8x8 head GEMM runs (0 = default). Allocates all
 * device scratch up front. */
int hn_create(hn_handle** out, int chunk_patches, long long head_rows);
int hn_destroy(hn_handle* h);

/* ---- HardNet (hardnet/HardNet.py:275-315) --------------------------------------------------------- */
/* Folds eval-mode BatchNorm (affine=False) into the conv weights and packs them K-major 16-bit.
 * HOST pointers: w[i] is features.{0,3,6,9,12,15,19}.weight in PyTorch OIHW order, bn_mean / bn_var the
 * matching running statistics of features.{1,4,7,10,13,16,20}. act_dtype: HN_F16 (default, 10-bit
 * mantissa like TF32) or HN_BF16. */
int hn_pack_hardnet(hn_handle* h, const float* const w[7], const float* const bn_mean[7],
                    const float* const bn_var[7], float bn_eps, int act_dtype);

/* The two epsilons of the forward: `input_norm_eps` is added to the per-patch std (1e-7 in hardnet/HardNet.py:309, 1e-8 in
 * HardNetNeiMask.input_norm, FDLNet-master/latency/rfnet/model/rf_des.py:41-49), `l2_eps` goes under the root of the final
 * L2 normalisation (1e-10 in hardnet/Utils.py:18; 0 for HardNetNeiMask's x / torch.norm(x), rf_des.py:51-55).
 * Defaults are HardNet's; the setting stays with the handle. */
int hn_set_hardnet_eps(hn_handle* h, float input_norm_eps, float l2_eps);

/* HardNet.forward in eval mode: input_norm -> 7 conv/BN/ReLU stages -> L2Norm.
 * patches: [B,1,32,32] (HN_F32 or HN_U8); desc_out: [B,128] (HN_F32 / HN_F16 / HN_BF16 / HN_F8E4M3). Every output dtype is the
 * fp32 descriptor rounded to nearest even (HN_F8E4M3: 128 bytes per row, equal to .to(torch.float8_e4m3fn) of the fp32 output). */
int hn_forward(hn_handle* h, const void* patches, int in_dtype, long long B, void* desc_out,
               int out_dtype, void* stream);

/* Test hook: run the stack up to and including conv stage `layer` (1..6) for B <= chunk_patches and
 * copy that stage's 16-bit activations to act_out in the device layout: stage 1 NHWC [B,H,W,C]; stages 2..6
 * channel-planar [B][C/8][H][W][8], where stages 2 and 4 (inputs of the stride-2 convs) hold the four
 * row/column parity sub-planes [B][C/8][ypar][xpar][H/2][W/2][8] (DESIGN.md section 3). */
int hn_forward_dump(hn_handle* h, const void* patches, int in_dtype, long long B, int layer,
                    void* act_out, void* stream);

/* Measurement hooks: bracket every launch of the selected stages (bit 0 = stage 1 alone (dump path only),
 * bit 1 = fused front kernel = stages 1 + 2, bits 2..5 = stages 3..6, bit 6 = head GEMM) with CUDA events on the launching stream; hn_profile_read waits for them, returns the
 * summed milliseconds and launch counts per stage and resets the counters. */
int hn_profile_enable(hn_handle* h, unsigned stage_mask);
int hn_profile_read(hn_handle* h, double ms_out[7], long long launches_out[7]);

/* ---- NAS-derived descriptor nets (hardnetNAS/fbnet_building_blocks, model_supernet.py:57-58,64-68,84) ------ */
/* One entry of the flat op list a sampled net is compiled to (hardnetnas_b200/nas/descriptor_net.py does the
 * compilation from the nn.Module tree: BatchNorm folded, channel shuffle folded into the producing 1x1 conv,
 * grouped 1x1 convs expanded to block-diagonal dense matrices). Activations live in three NHWC 16-bit slots. */
enum { HN_NAS_STEM = 0, HN_NAS_PW = 1, HN_NAS_DW = 2, HN_NAS_MAXPOOL = 3, HN_NAS_SE = 4, HN_NAS_HEAD = 5 };
typedef struct hn_nas_op {
  int kind;           /* HN_NAS_* */
  int cin, cout;      /* channels */
  int kernel, stride; /* DW: 3|5, 1|2; HEAD: kernel == hin */
  int hin, hout;      /* square spatial size in / out */
  int relu;
  int src, dst, res;  /* activation slots 0..2; res = residual input of a PW op or -1; STEM src = -1, HEAD dst = -1 */
  int mid;            /* SE hidden width */
  long long w_off, b_off, w2_off, b2_off; /* float offsets into `params` (fp32):
      STEM  w[9][32] (tap-major), b[32]            PW    w[cout][cin] dense, b[cout]
      DW    w[k*k][C], b[C]                        SE    w1[mid][C], b1[mid], w2[C][mid], b2[C]
      HEAD  w[128][(y*k+x)*cin + c], b[128] */
} hn_nas_op;

/* ops / params are HOST memory. Replaces any previously packed NAS net of the handle. */
int hn_pack_nas(hn_handle* h, const hn_nas_op* ops, int n_ops, const float* params, long long n_params,
                int act_dtype);
/* Eval forward of the packed net: [B,1,32,32] patches -> [B,128] unit descriptors (y / ||y||, no eps). */
int hn_forward_nas(hn_handle* h, const void* patches, int in_dtype, long long B, void* desc_out,
                   int out_dtype, void* stream);

/* Execution plan of the packed net: runs of consecutive ops behind the front stage that execute as ONE warpgroup-per-patch
 * tail launch (activations stay in shared memory between the run's first load and last store; hardnetNAS
 * fbnet_builder.py:455-570, an IRFBlock's pw -> dw -> pwl [+x] [+SE] never leaves the SM). Writes up to `cap` entries of 4 ints
 * (first op, last op, patches in flight per CTA, 0) to `out` (HOST memory, may be NULL) and returns the number of runs (>= 0)
 * or a negative hn_status. Ops outside every run execute as one kernel each. */
int hn_nas_plan(hn_handle* h, int* out, int cap);

/* Test hook: run ops [0, op_index] for B <= chunk_patches and copy that op's NHWC 16-bit output ([B,H,W,C]). */
int hn_forward_nas_dump(hn_handle* h, const void* patches, int in_dtype, long long B, int op_index,
                        void* act_out, void* stream);

/* ---- distances, hardest-in-batch mining, matching ------------------------------------------------- */
/* Bytes of device workspace hn_dist_min / hn_loss_hardnet / hn_match need for the given sizes. */
long long hn_dist_workspace_bytes(long long Na, long long Np, int split);

/* Fused distance matrix + masking + row (and column) minima; the Na x Np matrix never reaches HBM.
 * a:[Na,128], p:[Np,128] fp32. Outputs (any may be NULL): pos[min(Na,Np)] = diagonal distances
 * (before masking), row_min[Na] / row_arg[Na], col_min[Np] / col_arg[Np] (HN_FLAG_SWAP).
 * Replaces distance_matrix_vector + the eye/mask/min sequence of hardnet/Losses.py:95-108. */
int hn_dist_min(const float* a, const float* p, long long Na, long long Np, int form, int flags,
                float* pos, float* row_min, int32_t* row_arg, float* col_min, int32_t* col_arg,
                void* workspace, long long workspace_bytes, void* stream);

/* hn_dist_min with the neighbour mask of HardNetNeiMask.loss as an input of the fused epilogue (HN_FLAG_NEI_MASK, Na == Np):
 * a_xy / p_xy are the [N,2] fp32 (x, y) keypoint coordinates of the items in the anchor / positive image
 * (anchor_kp[:, 1:3], positive_kp[:, 1:3]); element (i, j) gets +10 if i == j, +10 if |a_xy[i] - a_xy[j]| < nei_c and +10 if
 * |p_xy[i] - p_xy[j]| < nei_c, with the reference's distance arithmetic (math_utils.py:22-40). pos = diagonal before masking. */
int hn_dist_min_ex(const float* a, const float* p, long long Na, long long Np, int form, int flags, const float* a_xy,
                   const float* p_xy, float nei_c, float* pos, float* row_min, int32_t* row_arg, float* col_min,
                   int32_t* col_arg, void* workspace, long long workspace_bytes, void* stream);

/* loss_HardNet, batch_reduce='min', loss_type='triplet_margin' (hardnet/Losses.py:87-108,142-143,153;
 * hardnetNAS/general_functions/Losses.py:27-51 is the anchor_swap=1 case). loss_out: 1 float (device). */
int hn_loss_hardnet(const float* anchor, const float* positive, long long N, float margin,
                    int anchor_swap, float* loss_out, void* workspace, long long workspace_bytes,
                    void* stream);

/* Brute-force matching in the FDLNet distance form: for every query row the nearest and second nearest
 * gallery rows (D.min(dim=-1) of eval_utils.py:113-114 and sorted[:,0:2] of :168-175).
 * q:[Nq,128], g:[Ng,128] fp32. Outputs: d1[Nq], d2[Nq] distances, i1[Nq] gallery index (+g_offset).
 * Requires g_offset >= 0 and Ng + g_offset < 2^31. A missing second neighbour (Ng == 1) is i2 = -1 whatever the offset.
 * Precondition: L2-normalised rows (|x| <= 1 up to rounding), the only input the FDLNet distance form is defined for
 * (math_utils.py:15-18 clamps 2 - 2ab to [1e-8, 4]): the exactness guarantee of the shortlist + fp32 re-rank rests on the
 * 2^-10 error bound of the fp16-operand dot product of unit vectors, and |x| >= 256 would overflow the packed operands. */
int hn_match(const float* q, const float* g, long long Nq, long long Ng, long long g_offset, float* d1,
             float* d2, int32_t* i1, int32_t* i2, void* workspace, long long workspace_bytes,
             void* stream);

/* The fp16 operand rows hn_match feeds to the tensor core (x * 2^8, K = 128), for callers that exchange the PACKED gallery
 * between GPUs (half the NVLink bytes of the fp32 rows) or match one set several times. x:[n,128] fp32 -> out16:[n,128]. */
int hn_pack_descriptors(const float* x, long long n, void* out16, void* stream);

/* Push all-gather of a gallery shard over NVSwitch multicast: packs x:[n,128] like hn_pack_descriptors and writes the packed
 * fp16 rows to mc16 and the fp32 rows to mc32, which must be MULTICAST addresses of symmetric buffers mapped on every GPU
 * of the group (e.g. torch.distributed._symmetric_memory: handle.multicast_ptr + this rank's row offset). The switch
 * replicates each store to all GPUs; after a cross-GPU barrier every GPU's local view of the buffers holds all shards.
 * Either destination may be NULL: the packed rows go first (the GEMM waits for them), the fp32 rows follow on a side stream
 * and land behind the GEMM (only the re-rank reads them). */
int hn_pack_descriptors_multicast(const float* x, long long n, void* mc16, void* mc32, void* stream);

/* hn_match with optional pre-packed operands (q16 / g16 from hn_pack_descriptors, NULL = pack here), an optional output of
 * the GEMM's block maxima (see hn_match_mutual; NULL = not computed) and an optional cudaEvent_t the exact re-rank waits for:
 * the GEMM reads only the packed rows, the re-rank reads the fp32 gallery rows of the shortlisted columns, so a sharded
 * caller gathers the packed gallery first and lets the fp32 gather finish behind the GEMM (hardnetnas_b200/distributed.py).
 * Preconditions as hn_match: unit-norm rows (|x| <= 1). */
int hn_match_ex(const float* q, const float* g, const void* q16, const void* g16, long long Nq, long long Ng,
                long long g_offset, float* d1, float* d2, int32_t* i1, int32_t* i2, float* block_max, void* workspace,
                long long workspace_bytes, void* g_ready_event, void* stream);

/* Mutual nearest neighbours from ONE matching GEMM (a16; composition of the reference's row / column minima,
 * hardnet/Losses.py:105-108, FDLNet-master/utils/eval_utils.py:24-32): mutual[i] = 1 iff i1[i] = argmin_j D[i,:] and
 * i = argmin_i D[:, i1[i]] (lowest index wins ties in both directions, like torch.min).
 * The row side is hn_match. For the column side the GEMM epilogue also emits `block_max`
 * [ceil(Ng/8)][ceil(Nq/32)]: the maximum approximate dot product of every (32-query block, 8-gallery-column chunk) cell.
 * Then (1) every query claims its nearest column (packed (distance, row) atomicMin: only the best claimant can be mutual),
 * (2) one warp per column chunk checks in exact fp32 the few cells that can still hold a closer query than the claimant: the
 * cell's maximum must reach the claimant's dot product AND some row of the cell must have its own second-nearest distance
 * d2 <= the claimant's distance (any other column of that row is at least d2 away) - confident matches are never challenged,
 * (3) mutual[i] = I hold the claim and it was not beaten. Distances are summed in the re-rank's order, so the result equals two hn_match passes bit for bit
 * wherever both shortlists are exact. d1 / d2 / i1 / i2 as hn_match (d1, i1, mutual required). */
long long hn_mutual_workspace_bytes(long long Nq, long long Ng);
int hn_match_mutual(const float* q, const float* g, const void* q16, const void* g16, long long Nq, long long Ng, float* d1,
                    float* d2, int32_t* i1, int32_t* i2, unsigned char* mutual, void* workspace, long long workspace_bytes,
                    void* stream);
/* The column-side steps on their own, for the sharded form (each rank holds a block of query rows starting at global row
 * q_offset and the whole gallery): claims of the local rows into `claim` [Ng] (initialised to INT64_MAX = unclaimed;
 * all_reduce(MIN) as int64 across ranks afterwards), then verification of the GLOBAL claims against the local rows with the block maxima of the
 * local hn_match_ex call into `beaten` [Ng] (initialised to 0; all_reduce(MAX) afterwards). Both require q_offset >= 0 and
 * Nq + q_offset < 2^32: the claims hold the global row as an unsigned 32-bit id, so the largest row id is 2^32 - 2. */
long long hn_block_max_elems(long long Nq, long long Ng);
int hn_mutual_claims(const int32_t* i1, const float* d1, const float* d2, long long Nq, long long q_offset,
                     unsigned long long* claim, long long Ng, float* rb_min_d2 /*[ceil(Nq/32)] out*/, void* stream);
int hn_mutual_verify(const float* q, long long Nq, long long q_offset, const float* g, long long Ng,
                     const unsigned long long* claim, const float* block_max, const float* rb_min_d2, unsigned char* beaten,
                     void* stream);

/* Batched matching: B independent problems of the shapes hn_match / hn_match_mutual solve, in one launch sequence (the shape
 * of an evaluation loop over image pairs, FDLNet-master/utils/eval_utils.py:85-197). q:[B,Nq,128], g:[B,Ng,128] fp32 padded
 * batches with unit-norm rows; q_len / g_len: DEVICE int32 [B] valid row counts per pair (NULL = all rows), clamped to
 * [0, Nq] / [0, Ng] on the device, so the call reads nothing on the host and is CUDA-graph capturable.
 * Outputs [B*Nq]: for a valid row r < q_len[b], d1 / d2 / i1 / i2 equal hn_match(q[b, :q_len[b]], g[b, :g_len[b]]) bit for bit
 * (indices local to the pair) and mutual (optional, NULL = no column side) equals hn_match_mutual on the same slices, wherever
 * the shortlists are exact (see hn_match). Rows past q_len[b], and every row of a pair with g_len[b] == 0, get d1 = d2 = +inf,
 * i1 = i2 = -1 and mutual = 0; g_len[b] == 1 gives d2 = +inf, i2 = -1. Padding rows may hold anything (NaN included): they
 * never influence another row or pair. Requires B*Nq and B*Ng below 2^31 and a 256-byte-aligned workspace of
 * hn_match_batched_workspace_bytes(B, Nq, Ng, mutual != NULL) bytes. */
long long hn_match_batched_workspace_bytes(long long B, long long Nq, long long Ng, int with_mutual);
int hn_match_batched(const float* q, const float* g, long long B, long long Nq, long long Ng, const int32_t* q_len,
                     const int32_t* g_len, float* d1, float* d2, int32_t* i1, int32_t* i2, unsigned char* mutual,
                     void* workspace, long long workspace_bytes, void* stream);

/* Pair-table matching: B problems over row ranges of two concatenated descriptor sets, in the launch sequence of
 * hn_match_batched. q:[Nq_rows,128], g:[Ng_rows,128] fp32 unit rows (the
 * descriptors of several images, concatenated); q16 / g16 their packed rows from hn_pack_descriptors (required, 16-byte
 * aligned; q may be g and q16 may be g16). pairs: DEVICE int32 [B][4] = (q_start, q_len, g_start, g_len): pair b matches rows
 * [q_start, q_start + q_len) of q against rows [g_start, g_start + g_len) of g. Clamped on the device: start to [0, N_rows];
 * len to [0, min(max_q or max_g, N_rows - start)]. The host never reads the table, so the call is CUDA-graph capturable and
 * a captured graph follows edits of the table.
 * Outputs are padded per pair like hn_match_batched: d1/d2/i1/i2[/mutual] [B*max_q], row r of pair b at b*max_q + r; for a
 * valid row they equal hn_match / hn_match_mutual on the two slices bit for bit (indices local to the pair's gallery range);
 * rows past q_len, and every row of a pair with g_len == 0, get +inf / -1 / 0. Rows outside a pair's ranges never influence
 * it. Requires Nq_rows, Ng_rows, B*max_q and B*max_g below 2^31 and a 256-byte-aligned workspace of
 * hn_match_pairs_workspace_bytes(B, max_q, max_g, mutual != NULL) bytes (it does not depend on the set sizes). */
long long hn_match_pairs_workspace_bytes(long long B, long long max_q, long long max_g, int with_mutual);
int hn_match_pairs(const float* q, const void* q16, long long Nq_rows, const float* g, const void* g16, long long Ng_rows,
                   const int32_t* pairs, long long B, long long max_q, long long max_g,
                   float* d1, float* d2, int32_t* i1, int32_t* i2, unsigned char* mutual,
                   void* workspace, long long workspace_bytes, void* stream);

/* Test / measurement switch (process-wide): which matching GEMM hn_match runs: -1 = chosen by problem size (default; the
 * initial value is read once from HN_MATCH_PAIR), 0 = single-CTA kernel, 1 = CTA-pair (cta_group::2) kernel. */
int hn_match_force_kernel(int mode);

/* ---- matching on fp16 / bf16 / fp8 E4M3 descriptor rows --------------------------------------------------------------------
 * Typed twins of the row-reading matching entry points: descriptor rows are `const void*` of desc_dtype HN_F32, HN_F16 or
 * HN_BF16 (e.g. the out_dtype output of hn_forward / hn_forward_nas / hn_forward_clip), the same type on both sides of a call;
 * the other arguments, the outputs and the preconditions are those of the fp32 function named. Every kernel widens a 16-bit
 * element to fp32 where it loads it and then runs the fp32 arithmetic: the packed operand is __float2half_rn(float(x) * 2^8)
 * as for fp32 rows, and the re-rank and the mutual verification sum the same fp32 products in the same order. So a call on
 * 16-bit rows returns exactly what the fp32 call returns on the rows converted to fp32 (distances, indices, ties, mutual
 * flags, bit for bit), without that fp32 copy: the re-rank and verification read 256 instead of 512 bytes per row.
 * The workspace does not depend on the row type: hn_dist_workspace_bytes, hn_mutual_workspace_bytes,
 * hn_match_batched_workspace_bytes and hn_match_pairs_workspace_bytes size the typed calls too. Validation as the fp32
 * function, plus: a desc_dtype other than HN_F32 / HN_F16 / HN_BF16 (HN_U8 included) and 16-bit rows that are not 8-byte
 * aligned are rejected with HN_ERR_INVALID before any device work. The fp32 functions are these calls with HN_F32.
 * HN_F8E4M3 rows (128 bytes per row, 4-byte aligned) follow the same contract: every output equals the fp32 call on the rows
 * converted to fp32, bit for bit. Their packed operand is e4m3 x * 2^8 ([n,128], 128 bytes per row), which is exact: a row
 * element of a unit row has |x| <= 1, so |x * 2^8| <= 256 < 448, and the smallest e4m3 subnormal 2^-9 becomes the normal
 * 2^-1. The matching GEMM then runs on the fp8 tensor core (kind::f8f6f4); its products are exact and only the accumulation can
 * differ from the fp16 GEMM (dist.cu states the bound the re-rank and verification margins rely on). Packed operands given by the
 * caller (q16 / g16) must come from hn_pack_descriptors_typed on rows of the call's dtype: e4m3 for HN_F8E4M3 rows, fp16
 * otherwise; the Python wrappers check this. An fp8 call needs no more workspace than the fp32 call the *_workspace_bytes
 * functions size. hn_pack_descriptors_multicast, hn_dist_min and hn_loss_hardnet take fp32 rows only. */
int hn_pack_descriptors_typed(const void* x, int desc_dtype, long long n, void* out16, void* stream);          /* hn_pack_descriptors */
int hn_match_typed(const void* q, const void* g, int desc_dtype, const void* q16, const void* g16, long long Nq, long long Ng,
                   long long g_offset, float* d1, float* d2, int32_t* i1, int32_t* i2, float* block_max, void* workspace,
                   long long workspace_bytes, void* g_ready_event, void* stream);                              /* hn_match_ex */
int hn_match_mutual_typed(const void* q, const void* g, int desc_dtype, const void* q16, const void* g16, long long Nq,
                          long long Ng, float* d1, float* d2, int32_t* i1, int32_t* i2, unsigned char* mutual, void* workspace,
                          long long workspace_bytes, void* stream);                                            /* hn_match_mutual */
int hn_match_batched_typed(const void* q, const void* g, int desc_dtype, long long B, long long Nq, long long Ng,
                           const int32_t* q_len, const int32_t* g_len, float* d1, float* d2, int32_t* i1, int32_t* i2,
                           unsigned char* mutual, void* workspace, long long workspace_bytes, void* stream);  /* hn_match_batched */
int hn_match_pairs_typed(const void* q, const void* q16, long long Nq_rows, const void* g, const void* g16, long long Ng_rows,
                         int desc_dtype, const int32_t* pairs, long long B, long long max_q, long long max_g, float* d1, float* d2,
                         int32_t* i1, int32_t* i2, unsigned char* mutual, void* workspace, long long workspace_bytes,
                         void* stream);                                                                        /* hn_match_pairs */

/* ---- k nearest neighbours -------------------------------------------------------------------------------------------------
 * The k <= 8 gallery rows nearest to every query row in the FDLNet distance sqrt(clamp(2 - 2ab, 1e-8, 4)), sorted ascending
 * by (distance, gallery index): the first k columns of the reference's full row sort (FDLNet-master/utils/eval_utils.py:168-175,
 * `D.sort(dim=-1)`) without the Nq x Ng matrix. dist / idx are [rows][k]; a row with fewer than k gallery rows gets +inf / -1
 * in the missing slots. Distances are the re-rank's fp32 arithmetic, bit-identical to what hn_match reports for the same
 * (row, column). The result is always exact: it equals a brute-force fp32 evaluation of every column with that arithmetic
 * followed by a stable sort, whatever the ties (hn_match's five-chunk limit does not apply; dist.cu gives the argument).
 * k outside [1, 8] is rejected with HN_ERR_INVALID before any device work. Rows, dtypes (HN_F32 / HN_F16 / HN_BF16 /
 * HN_F8E4M3, bit for bit the fp32 call on the rows converted to fp32), packed operands and validation are those of
 * hn_match_typed (single problem, no g_offset) and hn_match_pairs_typed (pair table: indices local to the pair's gallery range,
 * rows past q_len and pairs with g_len == 0 get +inf / -1, CUDA-graph capturable). A padded batch q [B, Nq, 128], g [B, Ng, 128]
 * with lengths q_len / g_len is the pair table (b*Nq, q_len[b], b*Ng, g_len[b]) over the flattened [B*Nq] / [B*Ng] rows.
 * The workspace (256-byte aligned) is sized by the two *_topk_workspace_bytes functions. */
long long hn_match_topk_workspace_bytes(long long Nq, long long Ng);
int hn_match_topk_typed(const void* q, const void* g, int desc_dtype, const void* q16, const void* g16, long long Nq, long long Ng,
                        int k, float* dist, int32_t* idx, void* workspace, long long workspace_bytes, void* stream);
long long hn_match_pairs_topk_workspace_bytes(long long B, long long max_q, long long max_g);
int hn_match_pairs_topk_typed(const void* q, const void* q16, long long Nq_rows, const void* g, const void* g16, long long Ng_rows,
                              int desc_dtype, const int32_t* pairs, long long B, long long max_q, long long max_g, int k,
                              float* dist, int32_t* idx, void* workspace, long long workspace_bytes, void* stream);

/* ---- radius matching ------------------------------------------------------------------------------------------------------
 * Every gallery row closer than `radius` to each query row: the entries of row i are the columns j with d(i, j) < radius
 * (strict, like D.lt(radius)), d the FDLNet distance in the re-rank's fp32 arithmetic, bit-identical to what hn_match /
 * hn_match_topk_typed report for the same (row, column). The result is exact: it equals a brute-force fp32 evaluation of every
 * column with that arithmetic (dist.cu gives the argument). Output is CSR: row_ptr int64 [rows + 1] (row_ptr[0] = 0,
 * row_ptr[rows] = nnz, up to rows * Ng), col int32 [capacity] and optional dist fp32 [capacity]; within a row the columns
 * ascend, so the flattened entries are in the row-major order of D.lt(radius).nonzero() and feed torch.sparse_csr_tensor as
 * they are. radius <= sqrtf(1e-8f) (about 1e-4; the clamp keeps every d at or above it) gives no entries, radius > 2 every
 * column; all-zero rows are at d = sqrt(2) from every column.
 * Two phases, as the output size is unknown in advance:
 *   1. count: packing, the top-k GEMM, a counting re-rank and an exclusive scan into row_ptr;
 *   2. fill: writes every entry whose CSR position is below `capacity` (nothing at or past it; row_ptr[rows] > capacity means
 *      the output was truncated). dist may be NULL; col may be NULL when capacity is 0.
 * The fill reads the candidate lists the count left in the workspace: call it with the same rows, table and radius, on the same
 * stream, with nothing run on the workspace in between. Neither phase reads anything on the host or allocates, so count + fill
 * with a known capacity is CUDA-graph capturable (and a captured pair-table graph follows edits of the table).
 * Rows, dtypes (HN_F32 / HN_F16 / HN_BF16 / HN_F8E4M3, bit for bit the fp32 call on the rows converted to fp32), packed operands
 * and validation are those of hn_match_topk_typed and hn_match_pairs_topk_typed. Pair tables: rows are the [B * max_q] padded
 * rows (row r of pair b at b * max_q + r), col is local to the pair's gallery range, rows past q_len and pairs with g_len == 0
 * have no entries. Also rejected with HN_ERR_INVALID before any device work: a NaN radius, capacity < 0, col == NULL with
 * capacity > 0, a row_ptr that is not 8-byte aligned, col / dist that are not 4-byte aligned, a workspace (256-byte aligned)
 * smaller than the *_radius_workspace_bytes function gives. */
long long hn_match_radius_workspace_bytes(long long Nq, long long Ng);
int hn_match_radius_count_typed(const void* q, const void* g, int desc_dtype, const void* q16, const void* g16, long long Nq,
                                long long Ng, float radius, long long* row_ptr, void* workspace, long long workspace_bytes,
                                void* stream);
int hn_match_radius_fill_typed(const void* q, const void* g, int desc_dtype, long long Nq, long long Ng, float radius,
                               const long long* row_ptr, long long capacity, int32_t* col, float* dist, void* workspace,
                               long long workspace_bytes, void* stream);
long long hn_match_pairs_radius_workspace_bytes(long long B, long long max_q, long long max_g);
int hn_match_pairs_radius_count_typed(const void* q, const void* q16, long long Nq_rows, const void* g, const void* g16,
                                      long long Ng_rows, int desc_dtype, const int32_t* pairs, long long B, long long max_q,
                                      long long max_g, float radius, long long* row_ptr, void* workspace, long long workspace_bytes,
                                      void* stream);
int hn_match_pairs_radius_fill_typed(const void* q, const void* q16, long long Nq_rows, const void* g, const void* g16,
                                     long long Ng_rows, int desc_dtype, const int32_t* pairs, long long B, long long max_q,
                                     long long max_g, float radius, const long long* row_ptr, long long capacity, int32_t* col,
                                     float* dist, void* workspace, long long workspace_bytes, void* stream);

/* Measurement hooks (process-wide): bracket the three stages of every hn_match / hn_match_batched / hn_match_pairs /
 * hn_match_topk_typed / hn_match_pairs_topk_typed call and of the radius calls (0 = operand packing, not part of the pair-table
 * calls; 1 = GEMM + shortlist, the count phase only; 2 = exact re-rank: the count re-rank with its scan, and the fill re-rank)
 * with CUDA events; hn_match_profile_read waits for them, returns the summed milliseconds and launch counts per stage and
 * resets the counters. */
int hn_match_profile_enable(int on);
int hn_match_profile_read(double ms_out[3], long long launches_out[3]);
/* Count of the top-k rows, and of the rows of radius count phases, whose re-rank scanned a whole candidate list because the
 * list's dropped maximum reached the threshold (process-wide, current device, off by default): enable(1) resets and starts it,
 * enable(0) stops it; read waits for the device, returns the count and resets it. */
int hn_match_topk_fallback_enable(int on);
int hn_match_topk_fallback_read(long long* rows_out);

/* ---- evaluation metrics of the test loop (hardnet/HardNet.py:443-477) -------------------------------------------------- */
/* Row-wise descriptor distance torch.sqrt(torch.sum((out_a - out_p) ** 2, 1)) (HardNet.py:458). a, p: [n,128] fp32; out: [n]. */
int hn_pair_distances(const float* a, const float* p, long long n, float* out, void* stream);
/* ErrorRateAt95Recall(labels, scores) (hardnet/EvalMetrics.py:6-19) without the host-side sort: the threshold element (the
 * ceil(0.95 * #positives)-th positive in ascending 1 / (scores + 1e-8) order, equal distances in input order like a stable
 * sort) is found by radix selection and the negatives in front of it are counted. scores: [n] fp32 = 1 / (distance + 1e-8)
 * as in HardNet.py:472; labels: [n] uint8 (non-zero = matching pair); out4 (DEVICE int64[4]) = FP, TN, #positives,
 * threshold_index. FPR95 = FP / (FP + TN). */
int hn_fpr95(const float* scores, const unsigned char* labels, long long n, long long* out4, void* stream);

/* ---- patch extraction (FDLNet-master/utils/image_utils.py:11-158, clip_patch) ------------------------ */
/* Crops a psize x psize patch around every keypoint with the reference's similarity transform
 * (scale / im_info[b][0] / 2, optional rotation (cos, sin)) and bilinear interpolation with clamped taps.
 * images [B,1,H,W] fp32; kpts_byxc [N,4] int64 (b, y, x, 0); kpts_scale [N]; kpts_ori [N,2] or NULL;
 * im_info [B,2]; out [N,1,psize,psize] fp32 (the input layout of hn_forward). N must be a multiple of B
 * (the reference reshapes the keypoints with view(B, -1)). */
int hn_clip_patches(const float* images, long long B, int H, int W, const long long* kpts_byxc,
                    const float* kpts_scale, const float* kpts_ori, const float* im_info, long long N,
                    int psize, float* out, void* stream);
/* hn_clip_patches (psize 32) + hn_forward in one call, with the crop done by the loader warps of the first conv kernel: the
 * [N,1,32,32] fp32 patch tensor never exists in device memory. Replaces the pair of calls in RFNetSO.inference
 * (FDLNet-master/latency/rfnet/model/rf_net_so.py:160-180: clip_patch(...) then self.des(patches)). images [B,1,H,W] of
 * img_dtype HN_F32 or HN_U8 (uint8 pixels are converted to fp32 before the interpolation, i.e. the result equals the fp32 call on
 * images.float()); keypoint arguments as hn_clip_patches; desc_out [N,128] of out_dtype. Descriptors are bit-identical to
 * hn_clip_patches followed by hn_forward. A keypoint whose image index is outside [0, B) yields a NaN descriptor. */
int hn_forward_clip(hn_handle* h, const void* images, int img_dtype, long long B, int H, int W, const long long* kpts_byxc,
                    const float* kpts_scale, const float* kpts_ori, const float* im_info, long long N, void* desc_out,
                    int out_dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HARDNET_B200_H_ */
