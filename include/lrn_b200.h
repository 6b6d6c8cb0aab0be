/*
 * lrn_b200.h -- C ABI of the B200-native (sm_100a) LineRefineNet forward hot path.
 *
 * The reference (1pathplanningzzj/pointnet_refine) has no native code on this
 * path: its "FFI" is whatever PyTorch dispatches for the ops in
 * src/model.py.  Each entry point below therefore cites the reference
 * *Python* interface it replaces (file:line in the reference tree).  The
 * reference-side binding (a ctypes stub) is shown in INTEGRATION.md; the
 * in-tree host mirror is pointnet_refine_b200/model.py.
 *
 * Conventions
 *   - All pointers are raw CUDA *device* pointers unless the name ends in
 *     "_host".  The caller owns every buffer, including the workspace (size
 *     via lrn_*_workspace_bytes); the library never allocates or frees device
 *     memory and never synchronises the device.
 *   - Every call is enqueued on the passed stream (cudaStream_t) and is
 *     stream-ordered and re-entrant; one host thread per process per GPU.
 *   - Return value: lrn_status (0 = ok).  No C++ exceptions cross the ABI.
 *     lrn_last_error() returns a thread-local detail string.
 *   - sm_100a only.  On any other device every compute call returns
 *     LRN_ERR_UNSUPPORTED_ARCH; there is no fallback path.
 */
#ifndef LRN_B200_H
#define LRN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* 2: lrn_train_attention_forward / _backward take `seed_state`; lrn_adam_step_capturable added
 * 3: lrn_launch_count added; later, without a version change, lrn_scenes_segments / lrn_scenes_workspace_bytes (lines of
 *    many scenes in one call).  Those are additions only: every entry point above keeps its signature and its results,
 *    so a caller built against an earlier version-3 library runs unchanged, and a caller that needs the additions finds
 *    them missing by name when it loads an older library (pointnet_refine_b200/_lib.py reports which).
 * 4: the per-scene segment builder and its workspace-size function removed: the lines of one scene are the K = 1 case
 *    of lrn_scenes_segments, which gives the same bits.
 * 5: the head gather of attention gradients and the host-counted lrn_adam_step removed: the train attention backward
 *    writes dK / dV in place in the K / V projections' layout, and every Adam step keeps its step count on the device
 *    (lrn_adam_step_capturable).  Later, without a version change, the output flag LRN_OUT_FUSED_BF16 of
 *    lrn_encoder_forward: an addition only; every flag combination that existed keeps its workspace size, its launches
 *    and its results.  A library built before it ignores the bit, so a call that requests nothing else fails there
 *    with LRN_ERR_BAD_ARG (no output requested). */
#define LRN_ABI_VERSION 5

typedef struct CUstream_st* lrn_stream_t; /* == cudaStream_t */

enum lrn_status {
  LRN_OK = 0,
  LRN_ERR_BAD_SHAPE = 1,        /* B/N/rows out of range                                  */
  LRN_ERR_MISALIGNED = 2,       /* a pointer is not 16-byte aligned                       */
  LRN_ERR_UNSUPPORTED_ARCH = 3, /* current device is not compute capability 10.0          */
  LRN_ERR_CUDA = 4,             /* a CUDA runtime/driver call failed (see lrn_last_error) */
  LRN_ERR_WORKSPACE = 5,        /* workspace/packed buffer too small                      */
  LRN_ERR_BAD_ARG = 6,          /* null required pointer, bad enum or flag combination    */
};

/* Arithmetic tier of the tensor-core layers (conv2..conv5, fusion, gate layer 2,
 * context_proj).  conv1 and gate layer 1 always run in fp32 FMA on raw fp32 xyz/intensity.
 *   BF16: operands rounded to bfloat16, fp32 accumulate  (tolerance 1e-2 of range)
 *   TF32: operands fp32 read as TF32, fp32 accumulate    (tolerance 1e-3 max-abs)
 *   FP32X3: every operand as two TF32 halves (hi + lo), three tensor-core passes per k-block (hi*hi + lo*hi + hi*lo), fp32
 *         accumulate, gate evaluated in full fp32: fp32-class products (relative error ~2^-21 per product) for callers that
 *         need the max-pool ARGMAX of the fp32 reference (src/model.py:58); about a third of the TF32 tier's throughput. */
enum lrn_precision { LRN_PREC_BF16 = 0, LRN_PREC_TF32 = 1, LRN_PREC_FP32X3 = 2 };

/* Output selection for lrn_encoder_forward (bitwise or). */
enum lrn_encoder_flags {
  LRN_OUT_POOL = 1,   /* global_feat (B,2048) = [max_n | mean_n]      src/model.py:58-60 */
  LRN_OUT_ARGMAX = 2, /* argmax (B,1024) int64, first index on ties   src/model.py:58 (torch.max indices) */
  LRN_OUT_FUSED = 4,  /* fused fp32 in the reference layout (B,1024,N) src/model.py:55,62 */
  LRN_OUT_MEMORY = 8, /* memory fp32 (B,N,256) = context_proj(fused^T) src/model.py:194   */
  LRN_OUT_MEMORY_BF16 = 16, /* with LRN_OUT_MEMORY (bf16 tier): memory is written as bf16 into rows of pitch 512
                               elements, columns [0,256); columns [256,512) are left to the caller (lrn_pos_hidden) */
  LRN_OUT_FUSED_BF16 = 32,  /* bf16 tier only, not with LRN_OUT_FUSED (both write through `fused`): fused as bf16 in
                               point-major order (B*N, 1024), the layout lrn_encoder_train_forward writes with
                               fused_point_major = 1 and context_proj consumes; each element is the bf16 rounding (to
                               nearest even) of the fp32 value LRN_OUT_FUSED writes.  On its own it launches no
                               context_proj GEMM, reads no proj_w and needs no workspace beyond the operand rows. */
};

/* Raw fp32 parameters of the reference module, exactly as they sit in its state_dict
 * (SURVEY.md appendix B).  Conv1d weights are (C_out, C_in, 1) contiguous == (C_out, C_in).
 * Replaces: MultiScalePointNetEncoder.__init__ parameter tree, src/model.py:7-37, and
 * LineRefineNet.context_proj, src/model.py:147. */
typedef struct lrn_encoder_params {
  const float* conv_w[5];   /* context_encoder.conv{1..5}.weight  (64,4) (128,64) (256,128) (512,256) (1024,512) */
  const float* conv_b[5];   /* context_encoder.conv{1..5}.bias                                   */
  const float* bn_w[5];     /* context_encoder.bn{1..5}.weight                                   */
  const float* bn_b[5];     /* context_encoder.bn{1..5}.bias                                     */
  const float* bn_mean[5];  /* context_encoder.bn{1..5}.running_mean                             */
  const float* bn_var[5];   /* context_encoder.bn{1..5}.running_var                              */
  const float* fusion_w;    /* context_encoder.fusion.0.weight (1024,1984)                       */
  const float* fusion_b;    /* context_encoder.fusion.0.bias                                     */
  const float* fusion_bn_w; /* context_encoder.fusion.1.{weight,bias,running_mean,running_var}   */
  const float* fusion_bn_b;
  const float* fusion_bn_mean;
  const float* fusion_bn_var;
  const float* gate0_w;     /* context_encoder.intensity_gate.0.weight (64,1)                    */
  const float* gate0_b;
  const float* gate2_w;     /* context_encoder.intensity_gate.2.weight (1024,64)                 */
  const float* gate2_b;
  const float* proj_w;      /* context_proj.weight (256,1024); may be NULL if LRN_OUT_MEMORY is never used */
  const float* proj_b;
  float bn_eps;             /* 1e-5 (torch.nn.BatchNorm1d default)                               */
} lrn_encoder_params;

/* ---- library / device ---- */
int lrn_abi_version(void);
const char* lrn_status_string(int status);
const char* lrn_last_error(void);
/* LRN_OK iff the current CUDA device can run this library (compute capability 10.0). */
int lrn_device_check(void);
/* Number of kernels this library has enqueued in this process (counted at enqueue: a CUDA-graph capture counts its
 * kernels once, replays of the graph count nothing). */
size_t lrn_launch_count(void);

/* ---- weight folding (eval-mode BatchNorm folded into the preceding 1x1 conv) ----
 * Replaces: the bn_k(conv_k(x)) pairs of MultiScalePointNetEncoder.forward in eval mode,
 * src/model.py:43-47,51 (W' = W*g/sqrt(var+eps), b' = (b-mean)*g/sqrt(var+eps)+beta), and
 * packs all matrices K-major in the tier's operand type.  Must be re-run whenever a
 * parameter or running statistic changes. */
size_t lrn_encoder_packed_bytes(int precision);
int lrn_encoder_fold(const lrn_encoder_params* params, int precision, void* packed, size_t packed_bytes,
                     lrn_stream_t stream);

/* ---- the hot path ----
 * Replaces: MultiScalePointNetEncoder.forward (src/model.py:39-62) in eval mode plus, with
 * LRN_OUT_MEMORY, the projection in LineRefineNet.forward (src/model.py:192-194).
 *   context      : (B, N, 4) fp32 contiguous [x,y,z,intensity] (the (B,4,N) view the module is
 *                  called with at src/model.py:192-193 is a transpose of this buffer)
 *   global_feat  : (B, 2048) fp32               required iff LRN_OUT_POOL or LRN_OUT_ARGMAX
 *   fused        : (B, 1024, N) fp32            required iff LRN_OUT_FUSED
 *                  ((B*N, 1024) bf16, 16-byte aligned, with LRN_OUT_FUSED_BF16; rows from B*N on are not written)
 *   argmax       : (B, 1024) int64              required iff LRN_OUT_ARGMAX
 *   memory       : (B, N, 256) fp32             required iff LRN_OUT_MEMORY  ((B, N, 512) bf16 with LRN_OUT_MEMORY_BF16)
 *   chunk_rows   : points processed per wave (0 = library default); a tuning knob only.
 * B >= 1, N >= 1, B*N < 2^31.  Empty input (B == 0 or N == 0) returns LRN_ERR_BAD_SHAPE, like
 * the reference, whose torch.max over an empty dimension raises. */
size_t lrn_encoder_workspace_bytes(int64_t B, int64_t N, int precision, int flags, int64_t chunk_rows);
int lrn_encoder_forward(const void* packed, int precision, const float* context, int64_t B, int64_t N, int flags,
                        float* global_feat, float* fused, int64_t* argmax, void* memory, int64_t chunk_rows,
                        void* workspace, size_t workspace_bytes, lrn_stream_t stream);

/* ---- point loading + first layer, stand-alone (tf32 tier, per-layer path, and bench.py's HBM roofline line) ----
 * Replaces: relu(bn1(conv1(x))) and the gate's Conv1d(1,64)+ReLU, src/model.py:43,33-34, in fp32 FMA on the raw points:
 * reads 16 B/point, writes feat1 -> operand columns [0,64) and the gate hidden block -> [1984,2048) of
 * `operand_rows` ((rows, 2048) in the tier's operand type).  HBM-bound: 16 + 256 B (bf16) / 16 + 512 B (tf32) per point.
 * tiled = 1 (bf16): `operand_rows` is in the tiled layout the default path keeps its operand matrix in,
 * [row tile of 128][column block of 64][128 rows][64 columns] (rows rounded up to 128): the two blocks a tile of points
 * writes are contiguous 16 KB pieces instead of 128-byte pieces at the 4 KB row pitch. */
int lrn_point_embed(const void* packed, int precision, const float* context, int64_t rows, void* operand_rows, int tiled,
                    lrn_stream_t stream);

/* ---- regression head + cumulative-offset bookkeeping ----
 * Replaces: reg_branches[i](tgt) and the coordinate update of LineRefineNet.forward,
 * src/model.py:172-179,220,227-231:
 *   delta = W2 relu(W1 tgt + b1) + b2;  current += delta;  cum_out = current - noisy
 *   w1 (128,256) b1 (128) w2 (3,128) b2 (3)  fp32 (reg_branches.{i}.{0,2}.{weight,bias})
 *   tgt (rows,256), current (rows,3) in/out, noisy (rows,3), cum_out (rows,3); rows = B*M. */
int lrn_head_forward(const float* w1, const float* b1, const float* w2, const float* b2, const float* tgt,
                     int64_t rows, float* current, const float* noisy, float* cum_out, lrn_stream_t stream);

/* ---- optional per-stage device timing (bench.py's roofline line) ----
 * New; nothing in the reference corresponds.  While enabled, lrn_encoder_forward brackets every
 * kernel it enqueues with cudaEvents on the caller's stream (events are owned by the library).
 * lrn_profile_read waits for the recorded events, returns the summed milliseconds and launch
 * counts per stage since the previous read, and resets.  Not thread-safe; off by default. */
enum lrn_stage {
  LRN_STAGE_EMBED = 0, /* conv1 + gate layer 1 (fp32 FMA, HBM-bound)  src/model.py:43,33-34 */
  LRN_STAGE_CONV2 = 1, /* src/model.py:44 */
  LRN_STAGE_CONV3 = 2, /* src/model.py:45 */
  LRN_STAGE_CONV4 = 3, /* src/model.py:46 */
  LRN_STAGE_CONV5 = 4, /* src/model.py:47 */
  LRN_STAGE_FUSION = 5,/* fusion conv + gate layer 2 + gating + pooling  src/model.py:50-60 */
  LRN_STAGE_PROJ = 6,  /* context_proj  src/model.py:194 */
  LRN_STAGE_COUNT = 7
};
int lrn_profile_enable(int on);
/* Tuning aid, only in the -DLRN_TIMELINE build (python pointnet_refine_b200/build.py --timeline; the product library
 * contains no timing code and returns LRN_ERR_BAD_ARG here): while `device_buffer` (>= 256 int64, zeroed by the caller) is
 * non-null, cluster 0 of the fusion / chain kernel records clock64() stamps of its first 16 tiles there (tools/timeline.py). */
int lrn_debug_timeline(long long* device_buffer);
int lrn_profile_read(float* ms_per_stage /*[LRN_STAGE_COUNT]*/, int64_t* launches_per_stage /*[LRN_STAGE_COUNT]*/);

/* ---- train mode: batch-statistic BatchNorm forward + hand-written backward of the context encoder ----
 * Replaces: MultiScalePointNetEncoder.forward under model.train() (src/model.py:39-55 with nn.BatchNorm1d in
 * training mode) and its autograd backward, as driven by train.py:56-72 / train_dist.py:168-189.  bf16
 * tensor-core operands, fp32 parameters and gradients.  context_proj stays with the caller (a differentiable
 * function of `fused`).
 *   global_feat : optional (fused_point_major = 0): (B, 2048) fp32 = [max_n | mean_n] of fused (src/model.py:58-60),
 *                 with argmax (B, 1024) int64 = first maximal point per (segment, channel).  The backward takes
 *                 d_global_feat + that argmax and scatters the max gradient to its argmax point / spreads the mean
 *                 gradient as 1/N inside its first kernel; d_fused may be NULL when only the pooled features carry
 *                 gradient (no dense (B,1024,N) gradient is built for the pooling).
 *   running     : running_mean / running_var of bn1..bn5 and fusion.1, updated in place like PyTorch
 *                 (momentum, unbiased variance); may be NULL.  num_batches_tracked is the caller's counter.
 *   fused       : fused_point_major = 0: (B,1024,N) fp32, the reference layout; 1: (B*N,1024) bf16 point-major
 *                 (what context_proj consumes, no layout change).  d_fused: its gradient, same layout / type.
 *   grads       : fp32 gradient of every encoder parameter (same shapes as lrn_encoder_params).
 *   workspace   : lrn_train_workspace_bytes(B, N); the forward leaves the saved activations there and the
 *                 matching backward call must receive the same, untouched buffer. */
typedef struct lrn_bn_running {
  float* mean[6]; /* bn1..bn5, fusion.1 */
  float* var[6];
} lrn_bn_running;
typedef struct lrn_encoder_grads {
  float* conv_w[5];
  float* conv_b[5];
  float* bn_w[5];
  float* bn_b[5];
  float* fusion_w;
  float* fusion_b;
  float* fusion_bn_w;
  float* fusion_bn_b;
  float* gate0_w;
  float* gate0_b;
  float* gate2_w;
  float* gate2_b;
} lrn_encoder_grads;
size_t lrn_train_workspace_bytes(int64_t B, int64_t N);
int lrn_encoder_train_forward(const lrn_encoder_params* params, const lrn_bn_running* running, float momentum,
                              const float* context, int64_t B, int64_t N, void* fused, int fused_point_major,
                              float* global_feat, int64_t* argmax, void* workspace, size_t workspace_bytes,
                              lrn_stream_t stream);
int lrn_encoder_train_backward(const lrn_encoder_params* params, const float* context, int64_t B, int64_t N,
                               const void* d_fused, int fused_point_major, const float* d_global_feat,
                               const int64_t* argmax, const lrn_encoder_grads* grads, void* workspace,
                               size_t workspace_bytes, lrn_stream_t stream);

/* ---- building block, exported for unit tests and profiling ----
 * out[M,N] = act(A[M,K] * W[N,K]^T + bias) on the tcgen05 tensor-core path.
 *   precision BF16: A, W bfloat16, out bfloat16 (out_f32 = 0) or fp32 (out_f32 = 1)
 *   precision TF32: A, W fp32,     out fp32 (out_f32 = 1) or bfloat16 (out_f32 = 0)
 * lda/ldw/ldo in elements; K % 64 == 0 (bf16) or K % 32 == 0 (tf32); N % 128 == 0. */
int lrn_gemm_bias_act(int precision, const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias,
                      void* out, int64_t ldo, int out_f32, int relu, int64_t M, int64_t N, int64_t K,
                      lrn_stream_t stream);

/* out[M,N] (fp32) = At^T * Bt with At (K, M) and Bt (K, N) bf16 row-major ("MN-major" tcgen05 operands): the
 * weight-gradient shape dW = dU^T X, K = points, read straight from the point-major buffers.  Few output tiles and a
 * long K are split over the CTA pairs (fp32 atomic accumulation into the zeroed output).
 * K % 64 == 0, M % 64 == 0, N % 128 == 0. */
int lrn_gemm_tn(const void* At, int64_t lda, const void* Bt, int64_t ldb, float* out, int64_t ldo, int64_t M, int64_t N,
                int64_t K, lrn_stream_t stream);

/* Cross attention of the 32 polyline queries of every segment over its N context points, all 8 heads, without
 * materialising K or V (replaces nn.MultiheadAttention cross_attn inside DetrTransformerDecoderLayer.forward,
 * src/model.py:123-128, for the eval path; SURVEY.md 8f row 1).
 *   qfold (B*256, 256) bf16: row h*32+q = log2(e)/sqrt(32) * (q_h[q] Wk_h), Wk_h = in_proj_weight[256+32h : 256+32h+32]
 *   kp    (B*N, 256)  bf16, row pitch ld_kp: memory + positional embedding     mem (B*N, 256) bf16, row pitch ld_mem: memory
 *   out   (B*splits*256, 256) fp32, or bf16 with out_bf16 = 1: softmax(qfold kp^T) mem per split, normalised inside the split
 *   lse   (B*splits*256) fp32: log2 of the split's sum of 2^score (to merge splits; splits = 1: final result)
 * The caller applies Wv_h / bv_h to `out` (rows of the softmax sum to one, so the bias passes through).
 * lrn_ctx_attention_splits(B, N) is the split count the library would pick (few segments: several clusters each). */
int lrn_ctx_attention_splits(int B, int N);
int lrn_ctx_attention(const void* qfold, const void* kp, int64_t ld_kp, const void* mem, int64_t ld_mem, int B, int N,
                      int splits, void* out, int out_bf16, float* lse, lrn_stream_t stream);

/* out[pt][0:256) = bf16(relu(W1 xyz + b1)): first layer of PositionalEncoding (src/model.py:66-75) on the context points
 * (context (P,4) fp32, xyz = first three columns; src/model.py:197).  out rows have a pitch of ld_out bf16 elements, so
 * it can fill columns [256,512) of the LRN_OUT_MEMORY_BF16 buffer: one GEMM with [I | W2] then yields memory + pos. */
int lrn_pos_hidden(const float* w1, const float* b1, const float* context, int64_t P, void* out, int64_t ld_out,
                   lrn_stream_t stream);

/* Parameter gradients of lrn_pos_hidden (train mode): d_w1 (256,3), d_b1 (256) fp32 (zeroed here) from the bf16 hidden
 * activations (ReLU mask) and their bf16 gradient, both (P, 256) with row pitches in elements. */
int lrn_pos_hidden_backward(const float* context, int64_t P, const void* hidden, int64_t ld_hidden, const void* d_hidden,
                            int64_t ld_d, float* d_w1, float* d_b1, lrn_stream_t stream);

/* resample_polyline (src/dataset.py:8-30) of L polylines to 32 and to 200 points on the device, bit-equal to the numpy
 * formulation: vertices (total, 3) f64 = all polylines back to back, offsets (L+1) int64 = first vertex of each line;
 * outputs line32 (L,32,3), dense200 (L,200,3), centers (L,3) f64 and noisy_centered (L,32,3) fp32 = line32 - center
 * (src/dataset.py:232-237).  A polyline with fewer than two vertices gives zeros; at most 2048 vertices per line. */
int lrn_scene_resample(const double* vertices, const int64_t* offsets, int L, int max_vertices, double* line32, double* dense200,
                       double* centers, float* noisy_centered, lrn_stream_t stream);
/* Scene preprocessing for L lines of K scenes in one call (SURVEY.md 8f row 3): the tube crop, weighted sampling and
 * centroid normalisation of LaneRefineDataset.__getitem__ steps 4-6 (src/dataset.py:214-237, weighted_sampling :78-130)
 * and of process_single_line (inference_whole_scene.py:95-121), which the reference runs on the host with one KD-tree per
 * line.  The lines of one scene are the case K = 1; lines of many scenes serve training batches that mix scenes and a
 * whole drive at inference.
 *   points    (S_total, 4) fp32 [x, y, z, intensity] device: K scenes back to back
 *   scene_offsets (K+1) int64 device: scene k is points[scene_offsets[k] .. scene_offsets[k+1])
 *   line_scene (L) int32: scene of every line, in the caller's order (lines of different scenes may be interleaved)
 *   dense200  (L, 200, 3) f64: resample_polyline(raw, 200)    line32  (L, 32, 3) f64: resample_polyline(raw, 32)
 *   centers   (L, 3) f64: mean of the 32 points                (all three as lrn_scene_resample writes them)
 *   seeds (L) uint64, line_ids (L) uint32: the RNG identity of every line
 *   context   (L, N, 4) fp32 out: sampled points, xyz - center (float64 subtraction, rounded once), intensity
 *   indices   (L, N) int64 out: index WITHIN the line's scene of every sample (-1: the zero points of an empty crop)
 *   counts    (L) int32 out: points inside the tube (distance to the 200-point polyline < crop_radius, float64 compare)
 *             (context, indices and counts in the caller's line order)
 *   status    (2) int64 out, one for the whole call: [0] total candidates, [1] bit 0: `capacity` < [0] -> nothing was
 *             sampled, call again with capacity >= status[0]; bit 1: more than 2^k - N candidates tie exactly at a line's
 *             threshold key; bit 2: some line_scene[l] is not in [0, K) (that line's outputs are not written)
 *   sorted_points / perm: optional (both or neither): every scene's points in a spatially coherent order (e.g. Morton order
 *             of x, y), concatenated as `points`, with perm[scene_offsets[k] + i] = index WITHIN scene k of
 *             sorted_points[scene_offsets[k] + i]; the crop then walks this copy, so that the 32 points of a warp are
 *             neighbours and only enter the tests of the lines that pass near them.  Results are identical.
 *   coord_extent: largest |coordinate| over the scenes and lines of the call.  It only sizes the band in which the fp32
 *             pre-filter defers to float64; the crop decision itself is exact for any extent at least that large (inside
 *             the band the distance is evaluated in double), so one extent per call gives the per-scene results.
 *   workspace at least lrn_scenes_workspace_bytes(L, K, capacity) bytes, 256-byte aligned; points / context 16-byte aligned
 * RNG: the draw of line l follows the RNG contract documented in oracle/scene_oracle.py (counter-based hash of seed, line,
 * scene index; Efraimidis-Spirakis keys; samples in descending key order) with (seed, line, scene index) = (seeds[l],
 * line_ids[l], index within scene line_scene[l]), i.e. scene_oracle.build_segment(scene_k, raw, N, r, decay, seeds[l],
 * line_ids[l]): same distribution as the reference's np.random.choice(replace=False, p), reproducible and independent of
 * thread order and of which lines share the call.
 * One pass: each point is tested only against the lines of its own scene; blocks of scenes without a line exit at once.
 * Launches per call are independent of K.  S_total < 2^31, K <= 65535, L <= 65535, N <= 4096 (else LRN_ERR_BAD_SHAPE). */
size_t lrn_scenes_workspace_bytes(int L, int K, int64_t capacity);
int lrn_scenes_segments(const float* points, const int64_t* scene_offsets, int K, int64_t S_total, const float* sorted_points,
                        const int32_t* perm, const int32_t* line_scene, const double* dense200, const double* line32,
                        const double* centers, const uint64_t* seeds, const uint32_t* line_ids, int L, int N, double crop_radius,
                        double decay_scale, double coord_extent, int64_t capacity, float* context, int64_t* indices, int32_t* counts,
                        int64_t* status, void* workspace, size_t workspace_bytes, lrn_stream_t stream);

/* ---- query side of the decoder (SURVEY.md 8f row 2; DetrTransformerDecoderLayer.forward, src/model.py:104-135) ----
 * out = LayerNorm(x + y) * gamma + beta over rows of 256 (norm1 / norm2 / norm3 with their residual adds, :117,:129,:134);
 * y may be NULL; cols must be 256 (d_model). */
int lrn_add_layernorm(const float* x, const float* y, const float* gamma, const float* beta, float eps, float* out,
                      float* stats /* optional (rows, 2): mean, rstd for the backward */, int64_t rows, int64_t cols,
                      lrn_stream_t stream);
/* Its backward (train mode): dz (rows,256) = gradient of x and of y, dgamma / dbeta (256) fp32 (zeroed here, then
 * accumulated); x, y, stats as in the forward call. */
int lrn_add_layernorm_backward(const float* dy, const float* x, const float* y, const float* stats, const float* gamma, float* dz,
                               float* dgamma, float* dbeta, int64_t rows, int64_t cols, lrn_stream_t stream);
/* Self attention over the 32 polyline points of each of B segments, 8 heads x 32 (self_attn, src/model.py:113-117, eval):
 * qk (B*32, 512) fp32 = [q | k] in-projections, v (B*32, 256) -> out (B*32, 256) heads concatenated (before out_proj). */
int lrn_self_attention32(const float* qk, const float* v, float* out, int B, lrn_stream_t stream);
/* Second layer of reg_branches[i] + the cumulative-offset update (src/model.py:220,227-231) for `rows` polyline points:
 * delta = hidden (rows,128) W2^T + b2; current += delta (in place); cum = current - noisy.  (lrn_head_forward does both
 * layers in one latency-oriented kernel; for thousands of rows layer 1 runs as a tensor-core GEMM and this finishes.) */
int lrn_head_update(const float* hidden, const float* w2, const float* b2, int64_t rows, float* current, const float* noisy,
                    float* cum, lrn_stream_t stream);

/* ---- query side for FEW polyline rows (B = 1 whole-scene calls, inference_whole_scene.py:130-139): one nn.Linear per launch,
 * fp32 FMA, the layer's weights read once and spread over N/8 blocks (a 256-row tensor-core tile would be mostly padding).
 *   out[M,N] = act(x'[M,K] w[N,K]^T + bias),  out fp32 or bf16 (out_bf16 = 1), relu optional, row pitches in elements.
 *   x' = x                      (x2 = NULL, mlp3_w1 = NULL)
 *   x' = x + x2                 (with_pos_embed: tgt + query_pos, src/model.py:101-102,113,124)
 *   x' = relu(mlp3_w1 c + mlp3_b1) with x = c (M,3): the K = 3 first layer of PositionalEncoding (src/model.py:68-72, called at
 *        :212) or of point_mlp (:151-153, BatchNorm folded by the caller) fused into the load of the second layer's operand.
 * Replaces the nn.Linear calls of DetrTransformerDecoderLayer.forward (src/model.py:104-135), pos_emb (:64-75) and
 * point_mlp (:150-159, 200-201) for query batches below 256 rows.  N % 8 == 0, K % 32 == 0. */
int lrn_rows_linear(const float* x, int64_t ldx, const float* x2, int64_t ldx2, const float* mlp3_w1, const float* mlp3_b1,
                    const float* w, const float* bias, void* out, int64_t ldo, int out_bf16, int relu, int64_t M, int64_t N,
                    int64_t K, lrn_stream_t stream);
/* out (rows,256) fp32 = relu(W1 c + b1): first layer of pos_emb (src/model.py:68-72) on the current polyline points (:212,
 * coords (rows,3), ld = 3) or on the context points (:197, coords = context (rows,4), ld = 4; tf32 tier) when the second
 * layer runs as a tensor-core GEMM.  round_tf32 = 1 rounds the result to the nearest TF32 value (a tf32-tier GEMM operand;
 * the tensor core would otherwise truncate it). */
int lrn_query_pos_hidden(const float* w1, const float* b1, const float* coords, int64_t ld, int64_t rows, float* out,
                         int round_tf32, lrn_stream_t stream);
/* out = a + b over n fp32 elements (n % 4 == 0): with_pos_embed ahead of a tensor-core linear.  b may be NULL (copy);
 * round_tf32 = 1 rounds the result to the nearest TF32 value. */
int lrn_add(const float* a, const float* b, float* out, int64_t n, int round_tf32, lrn_stream_t stream);
/* fp32 cross attention of the 32 polyline queries of each of B segments over its N context points, 8 heads x 32
 * (nn.MultiheadAttention cross_attn in eval mode, src/model.py:123-128; the tf32 tier, where K / V of all layers come from
 * hoisted TF32 GEMMs): q (B*32, 256) in-projected queries; k / v: point (b*N + n) at k + (b*N + n) * ld_kv (head h at
 * + 32 h), so a layer's K is a column block of the (B*N, L*256) GEMM result; out (B*32, 256) heads concatenated. */
int lrn_cross_attention32(const float* q, const float* k, const float* v, int64_t ld_kv, int B, int N, float* out,
                          lrn_stream_t stream);
/* Merge the splits of lrn_ctx_attention: part (B, splits, 256, 256) fp32, lse (B, splits, 256) -> out (B, 256, 256) fp32 or
 * bf16, out[b][q] = sum_s 2^(lse_s - max) part_s / sum_s 2^(lse_s - max). */
int lrn_ctx_attention_merge(const float* part, const float* lse, int B, int splits, void* out, int out_bf16, lrn_stream_t stream);

/* ---- train-mode attention for 32 queries per segment (nn.MultiheadAttention under model.train(): cross_attn over the N
 * context points, src/model.py:84,123-128, and self_attn over the 32 polyline points, :113-117; 8 heads x 32, dropout on the
 * attention weights).  K / V are read where the projections left them: key n of segment b at k + (b*N + n) * ld_k, head h at
 * + 32 h (for the cross attention pass a layer's column block of the (B, N, layers, 8, 32) bf16 projection buffer; ld_v
 * likewise).  q, out, dout, dq: (B, 32, 256) fp32, heads concatenated; lse (B, 8, 32) fp32 is written by the forward and
 * read by the backward.  The backward writes dk / dv for every key in the same addressing (row pitches ld_dk / ld_dv),
 * complete for this call: no per-head gradient tensors, no gathers.  Dropout: counter-based hash of (seed, segment, head,
 * query, key), regenerated by the backward; pass a fresh seed per call and the same one to its backward.  seed_state
 * (may be NULL) is a device word added to `seed` when the kernel runs: a captured CUDA graph (GraphedTrainStep) advances
 * that word inside the graph, so every replay draws a new mask although the launch arguments are frozen. */
int lrn_train_attention_forward(const float* q, const void* k, int64_t ld_k, const void* v, int64_t ld_v, int B, int N, float* out,
                                float* lse, float p_drop, uint64_t seed, const uint64_t* seed_state, lrn_stream_t stream);
int lrn_train_attention_backward(const float* q, const void* k, int64_t ld_k, const void* v, int64_t ld_v, int B, int N,
                                 const float* out, const float* lse, const float* dout, float* dq, void* dk, int64_t ld_dk, void* dv,
                                 int64_t ld_dv, float p_drop, uint64_t seed, const uint64_t* seed_state, lrn_stream_t stream);

/* out[c] = sum over rows of the bf16 matrix A (rows, cols), row pitch ld: the bias gradient of a linear layer whose output
 * gradient is bf16 (cols % 64 == 0, ld % 8 == 0, A 16-byte aligned). */
int lrn_col_sum_bf16(const void* A, int64_t ld, int64_t rows, int64_t cols, float* out, lrn_stream_t stream);

/* ---- training-loop machinery (SURVEY.md 8f row 4) ----
 * One Adam step over a flat fp32 buffer holding every parameter (train.py:40 optim.Adam(model.parameters(), lr);
 * torch.optim.Adam semantics without amsgrad, weight decay added to the gradient), with the step count kept on the
 * device (torch.optim.Adam(capturable=True) semantics): *step_state (0 before the first step) is incremented by a
 * one-thread kernel first and the bias corrections are computed from it on the device in double precision, so the two
 * launches can be captured in a CUDA graph and replayed (train.py:71 optimizer.step() inside GraphedTrainStep). */
int lrn_adam_step_capturable(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                             float beta2, float eps, float weight_decay, int64_t* step_state, lrn_stream_t stream);
/* Deep-supervision loss of train.py:63-69: loss[0] = (1/L) sum_l L1Loss(pred[l], target) for pred (L, n) and target (n)
 * (n = B*M*3 elements per decoder layer), and its gradient dpred (L, n) = sign(pred - target) / (L n); dpred may be NULL. */
int lrn_l1_deep_supervision(const float* pred, const float* target, int L, int64_t n, float* loss, float* dpred,
                            lrn_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* LRN_B200_H */
