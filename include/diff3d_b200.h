/*
 * diff3d_b200.h -- C ABI of libdiff3d_b200.so: the B200 (sm_100a) implementation of Diff3DHPE's
 * inference hot path (DDIM reverse sampling over the MixSTE seq2seq denoiser).
 *
 * The reference (csiro-icvg/Diff3DHPE) is pure Python/PyTorch and has no FFI layer; its seam is three
 * Python methods (SURVEY.md section 8b).  Each entry point below names the reference interface it
 * replaces, with file:line into the reference tree:
 *
 *   MODEL = common/nets/model_conditional_diffusion_mixste_s2s_grand_linLift.py
 *   DIFF  = common/conditional_diffusion_ddim_normal_directPredict_variableLoss_both_crossFrames.py
 *   RUN   = run_conditionalDiffusionDDIM3dhpeNormalDirectPredictVariableLoss.py
 *   LOSS  = common/loss.py
 *
 * Conventions
 *   - plain C types only; no C++ or torch types cross this boundary.
 *   - every function returns int: 0 = OK, negative = invalid argument / unsupported shape,
 *     positive = cudaError_t.  The message is available from d3d_last_error().  Nothing throws/exits.
 *   - all tensors are contiguous fp32, channel-last, exactly the reference's layouts:
 *     2D keypoints [B,F,J,2], poses [B,F,J,3], denoiser input [B,F,J,5].
 *   - "dev" pointers are device pointers on the handle's device, owned by the caller and valid until the
 *     work enqueued on `stream` has completed; "host" pointers are host memory (pinned for async copies).
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  All work is enqueued
 *     asynchronously on it unless stated otherwise.
 *   - a handle is bound to one device and is not thread-safe; use one handle per rank.
 *   - distinct handles may be created, used and destroyed concurrently from different threads, on the same
 *     device or on different ones (one thread per device is how nn.DataParallel drives the drop-in modules);
 *     one handle must not be used by two threads at once.  The library's process-wide state is limited to
 *     values initialised once, thread-safely, and the thread-local message of d3d_last_error(NULL).
 *   - the library owns packed weights, the time-embedding table, the activation workspace and its CUDA
 *     graphs; nothing is allocated on the hot path.
 */
#ifndef DIFF3D_B200_H_
#define DIFF3D_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define D3D_ABI_VERSION 1
#if defined(__GNUC__)
#define D3D_API __attribute__((visibility("default")))
#else
#define D3D_API
#endif

typedef struct d3d_handle d3d_handle;

/* GEMM arithmetic of the qkv/proj/fc1/fc2 linears (tcgen05.mma, fp32 accumulation in TMEM). */
enum {
  D3D_GEMM_TC_SPLIT3 = 0, /* 3-pass split-fp16 (a_hi*b_hi + a_hi*b_lo + a_lo*b_hi), ~fp32 accurate */
  D3D_GEMM_TC_FP16 = 1,   /* single-pass fp16 operands: fast mode, outside the 0.1 mm MPJPE-delta bar   */
  D3D_GEMM_SIMT_FP32 = 2, /* CUDA-core fp32 validation kernel (same operands as SPLIT3, no tensor cores) */
  D3D_GEMM_TC_F8C = 3,    /* default of the Python drop-ins: fp16 main product + one e5m2 (kind::f8f6f4) product carrying both correction terms:
                             2 tensor-pipe units instead of 3, within the parity bar (DESIGN.md section 2) */
  D3D_GEMM_SIMT_F8C = 4,  /* CUDA-core validation kernel on the F8C operand format */
  D3D_GEMM_TC_F4C = 5,    /* fp16 main product + one BLOCK-SCALED e2m1 product (kind::mxf4.block_scale, one ue8m0 scale per 32
                             elements of K, 4x the fp16 rate) carrying both correction terms: 1.5 tensor-pipe units, 3.06 operand
                             bytes per element */
  D3D_GEMM_SIMT_F4C = 6   /* CUDA-core validation kernel on the F4C operand format */
};
/* Attention kernels. */
enum {
  D3D_ATTN_DEFAULT = 0,   /* spatial: mma.sync smem/register kernel; temporal: tcgen05/TMEM/TMA kernel for F > 64,
                             mma.sync flash kernel for short sequences */
  D3D_ATTN_SIMT = 1,      /* CUDA-core fp32 validation kernels */
  D3D_ATTN_MMA_SYNC = 2   /* force the mma.sync (legacy tensor path) kernels for every F */
};

/* Mirrors the constructor of ConditionalDiffusionMixSTES2SGRANDLinLift (MODEL:140-142). */
typedef struct d3d_config {
  int32_t num_frame;     /* F: 27 / 81 / 243 (any 1..256)           */
  int32_t num_joints;    /* J: 17                                     */
  int32_t embed_dim;     /* C: 512 (kernels are specialised for 512)  */
  int32_t depth;         /* spatial/temporal block pairs: 8           */
  int32_t num_heads;     /* 8 (head_dim 64)                           */
  int32_t mlp_hidden;    /* int(C * mlp_ratio): 1024                  */
  int32_t with_time_emb; /* 0/1 (MODEL:163-177)                       */
  int32_t max_clips;     /* workspace capacity in clips (B)           */
  int32_t gemm_mode;     /* D3D_GEMM_*                                */
  int32_t attn_mode;     /* D3D_ATTN_*                                */
  int32_t device;        /* CUDA device ordinal                       */
  int32_t use_graph;     /* 1: replay the S-step loop as one CUDA graph */
} d3d_config;

/* One named fp32 parameter of the reference state dict ("fusion_layer.weight",
 * "STEblocks.3.attn.qkv.weight", ..., without the "module."/"model." prefixes). */
typedef struct d3d_tensor {
  const char* name;
  const float* data;
  int64_t numel;
  int32_t on_device; /* 0: host pointer, 1: device pointer on the handle's device */
} d3d_tensor;

D3D_API int d3d_abi_version(void);

/* Replaces the module constructor (MODEL:140-220): allocates workspace for max_clips clips. */
D3D_API int d3d_create(const d3d_config* cfg, d3d_handle** out);
D3D_API void d3d_destroy(d3d_handle* h);
/* Message of the last failing call on this handle (h == NULL: the calling thread's last failing d3d_create). */
D3D_API const char* d3d_last_error(const d3d_handle* h);

/* Replaces load_state_dict (RUN:226-235): copies, packs and (for GEMM operands) splits the weights.
 * Unknown names are an error; missing tensors are reported by the first call that needs them. */
D3D_API int d3d_load_weights(d3d_handle* h, const d3d_tensor* tensors, int32_t n);

/* Replaces the schedule part of GaussianDiffusion.__init__ / ddim_sample_loop (DIFF:119-183, 263-273,
 * 287-292).  times: S+1 entries (DIFF:270-272, last is -1); alphas_cumprod, sqrt_one_minus_alphas_cumprod:
 * the fp32 buffers of length T; eta: ddim_sampling_eta; clip_denoised: DIFF:252. */
D3D_API int d3d_set_schedule(d3d_handle* h, int32_t S, const int32_t* times, const float* alphas_cumprod,
                     const float* sqrt_one_minus_alphas_cumprod, int32_t T, float eta, int32_t clip_denoised);

/* Replaces model.forward_denoise (MODEL:249-257): x5 [B,F,J,5], t [B] (int64, per sample) -> out3 [B,F,J,3]. */
D3D_API int d3d_forward_denoise(d3d_handle* h, const float* x5_dev, const int64_t* t_dev, float* out3_dev, int32_t B,
                        void* stream);

/* Replaces GaussianDiffusion.ddim_sample_loop (DIFF:263-300) with the noise made explicit:
 *   noise0     [B,F,J,3]          the torch.randn of DIFF:275
 *   step_noise [S-1][B,F,J,3]     the randn_like of DIFF:293 per non-final step; may be NULL iff eta == 0
 *   y0         [B,F,J,3]          result
 *   trace_y / trace_x0            optional [B,F,J,3,S] stacks of DIFF:304-347 (NULL to skip). */
D3D_API int d3d_ddim_sample(d3d_handle* h, const float* x2d_dev, const float* noise0_dev, const float* step_noise_dev,
                    float* y0_dev, float* trace_y_dev, float* trace_x0_dev, int32_t B, void* stream);

/* Same, from/to HOST buffers (pinned): H2D copies, the sampler and the D2H copy are enqueued on `stream`
 * and the call returns after the stream has been synchronised.  This is the end-to-end entry point. */
D3D_API int d3d_ddim_sample_host(d3d_handle* h, const float* x2d_host, const float* noise0_host,
                         const float* step_noise_host, float* y0_host, int32_t B, void* stream);

/* Replaces the flip-TTA tail of evaluate() (RUN:583-588): out = (y + unflip(y_flip)) / 2 * scale, where
 * unflip negates x and swaps joints left[i] <-> right[i].  n_frames = B*F. */
D3D_API int d3d_tta_merge(d3d_handle* h, const float* y_dev, const float* y_flip_dev, const int32_t* joints_left,
                  const int32_t* joints_right, int32_t n_lr, float scale, float* out_dev, int64_t n_frames,
                  void* stream);

/* The remaining metrics of evaluate() (RUN:602-614) on the device ("next" row N4): for the n_sel frames listed in
 * frame_index_dev (NULL = frames 0..n_sel-1 in order) adds to acc_dev (six fp64 on the device)
 *   [0] sum_j ||pred - gt||                       mpjpe   (common/loss.py:15-27)
 *   [1] sum_j ||s pred - gt||, s per frame        n_mpjpe (common/loss.py:84-94)
 *   [2] sum_j ||procrustes(pred) - gt||           p_mpjpe (common/loss.py:43-82; 3x3 SVD per frame in fp64)
 *   [3] joints counted
 *   [4] sum over calls of n_sel * mean_velocity_error(this call's listed frames)   (common/loss.py:133-142: the mean runs
 *       over the (n_sel - 1) * J differences of consecutive listed frames), [5] sum over calls of n_sel -- the
 *       reference's own weighting, `epoch_loss_3d_vel += N_b * mean_velocity_error(batch)` over `N += N_b` (RUN:610-614)
 * pred_dev / gt_dev: [n_frames, J, 3].  mpjpe = [0]/[3], n_mpjpe = [1]/[3], p_mpjpe = [2]/[3], velocity = [4]/[5];
 * one call = one batch of evaluate(). */
D3D_API int d3d_pose_metrics_accumulate(d3d_handle* h, const float* pred_dev, const float* gt_dev,
                                const int64_t* frame_index_dev, int64_t n_sel, double* acc_dev, void* stream);

/* Windowing on the device (common/nosiy_generators.py:27-48, 264-276; "next" row N3 of SURVEY.md 8f).
 * seq2d_dev: packed sequences [n_frames_total, J, 2]; win_start_dev[w] = first packed frame of window w.  Writes
 * x2d_out_dev [n_win, F, J, 2] and, when x2d_flip_out_dev != NULL, the horizontally flipped copy (x negated, joints
 * left[i] <-> right[i] swapped) that the reference's generator hands to evaluate() as inputs_2d_flip. */
D3D_API int d3d_window_gather(d3d_handle* h, const float* seq2d_dev, const int64_t* win_start_dev, int64_t n_win,
                      const int32_t* joints_left, const int32_t* joints_right, int32_t n_lr, float* x2d_out_dev,
                      float* x2d_flip_out_dev, void* stream);

/* The inverse: writes pred_dev [n_win, F, J, 3] into packed per-sequence frame order seq3d_out_dev
 * [n_frames_total, J, 3], skipping the first first_valid_dev[w] frames of window w (target_mask of the back-shifted
 * last window of a sequence, nosiy_generators.py:264-271, applied by RUN:589-596). */
D3D_API int d3d_window_scatter(d3d_handle* h, const float* pred_dev, const int64_t* win_start_dev,
                       const int32_t* first_valid_dev, int64_t n_win, float* seq3d_out_dev, void* stream);

/* Replaces mpjpe (LOSS:15-27) + the N-weighted accumulation of RUN:602-606: adds sum_j ||pred-gt||_2 over the
 * frames whose mask byte is non-zero (mask NULL = all) to acc_dev[0] and the joint count to acc_dev[1]
 * (two fp64 on the device; MPJPE = acc[0]/acc[1]). */
D3D_API int d3d_mpjpe_accumulate(d3d_handle* h, const float* pred_dev, const float* gt_dev, const uint8_t* frame_mask_dev,
                         int64_t n_frames, double* acc_dev, void* stream);

/* Number of kernels launched (or replayed through graphs) by this handle since creation. */
D3D_API int64_t d3d_launch_count(const d3d_handle* h);

/* Device bytes the handle owns (packed weights, activation workspace, time tables, sampler state): everything is
 * allocated in d3d_create / d3d_set_schedule, nothing on the hot path (SURVEY.md 8b `d3d_workspace_bytes`).  16 KB per
 * token of max_clips * num_frame * num_joints + ~100 MB of weights: 34 GB for 512 clips of 243 frames. */
D3D_API int64_t d3d_workspace_bytes(const d3d_handle* h);

/* Per-kernel-class device timing.  Between d3d_profile_begin and d3d_profile_end every kernel of the sampler /
 * denoiser is launched un-graphed and bracketed by CUDA events on the launch stream; d3d_profile_end
 * synchronises and returns the summed durations (ms) and launch counts per class. */
enum {
  D3D_PROF_GEMM = 0,          /* qkv / proj / fc1 / fc2 tcgen05 GEMMs          */
  D3D_PROF_ATTN_SPATIAL = 1,  /* 17-joint attention                             */
  D3D_PROF_ATTN_TEMPORAL = 2, /* F-frame attention                              */
  D3D_PROF_LN = 3,            /* post-norm + add + norm1, norm2 (row-wise)      */
  D3D_PROF_LIFT = 4,          /* input lift + pos-embed + time vector + norm1   */
  D3D_PROF_HEAD = 5,          /* Temporal_norm + head + clamp + DDIM update     */
  D3D_PROF_NUM_CLASSES = 6
};
D3D_API int d3d_profile_begin(d3d_handle* h);
D3D_API int d3d_profile_end(d3d_handle* h, double* ms_per_class, int64_t* launches_per_class);

/* ---- kernel-level entry points (parity tests, microbenchmarks, ncu exhibits) ------------------------ */

/* out[M,N] = epilogue(A[M,K] . W[N,K]^T + bias[N]) with the handle's (or the given) GEMM mode.
 * act: 0 none, 1 exact-erf GELU.  residual (may be NULL) is added after the bias.  Operands are fp32 on the
 * device; the split into fp16 halves happens inside, as on the hot path.  K % 64 == 0, N % 128 == 0. */
D3D_API int d3d_op_linear(d3d_handle* h, const float* a_dev, const float* w_dev, const float* bias_dev,
                  const float* residual_dev, float* out_dev, int64_t M, int32_t N, int32_t K, int32_t act,
                  int32_t gemm_mode, void* stream);
/* Times `iters` back-to-back launches of the GEMM kernel alone (operands pre-split), returns ms/launch.
 * act: 0 fp32 output, 1 GELU -> operand, 2 fp32 output + in-place residual (proj / fc2 as they run in the step),
 * 3 = 2 + the emitted operand and row statistics of the deferred norm2 (N == 512), 4 = GELU with the deferred
 * LayerNorm applied in the epilogue (K == 512); 3 and 4 need D3D_GEMM_TC_F4C. */
D3D_API int d3d_op_linear_bench(d3d_handle* h, int64_t M, int32_t N, int32_t K, int32_t act, int32_t gemm_mode,
                        int32_t iters, float* ms_per_launch);

/* LayerNorm over the last dim (512): out = (x-mean)*rstd*gamma+beta (MODEL:184,218).  The per-row arithmetic is the
 * one of the hot path's row-wise kernels (two-pass variance, rsqrt + one Newton step, packed fp32 pairs), so `out` is
 * bit for bit the fp32 LayerNorm those kernels quantise into a GEMM operand. */
D3D_API int d3d_op_layernorm(d3d_handle* h, const float* x_dev, const float* gamma_dev, const float* beta_dev, float eps,
                     float* out_dev, int64_t rows, void* stream);

/* GRAND attention core (MODEL:76-83) on a packed qkv tensor [B*F*J, 3*C] (channel = which*C + head*64 + d):
 * spatial != 0: sequences are the J joints of a frame; else the F frames of a joint.  out: [B*F*J, C]. */
D3D_API int d3d_op_attention(d3d_handle* h, const float* qkv_dev, float* out_dev, int32_t B, int32_t spatial,
                     int32_t attn_mode, void* stream);

/* Time-embedding table (MODEL:29-36,169-174 and the per-block SiLU+Linear of MODEL:104-116):
 * t [R] (float) -> out [R, 2*depth, C]; block order STE0, TTE0, STE1, ... */
D3D_API int d3d_op_time_table(d3d_handle* h, const float* t_host, int32_t R, float* out_dev, void* stream);

/* Runs forward_denoise but stops after `n_blocks` transformer blocks (0..2*depth) and copies the fp32
 * residual stream [B*F*J, C] as it stands BEFORE the next post-norm into x_out_dev. */
D3D_API int d3d_debug_forward_blocks(d3d_handle* h, const float* x5_dev, const int64_t* t_dev, int32_t B,
                             int32_t n_blocks, float* x_out_dev, void* stream);

/* The fused "proj + residual + norm2" kernel (MODEL:127-128) on explicit operands: x_out = a . w^T + bias + residual
 * ([M,512], K = columns of a), ln_out = LayerNorm(x_out; gamma, beta, eps) read back from the operand format it is
 * written in (fp16 hi + e5m2 lo).  Needs gemm_mode D3D_GEMM_TC_F8C. */
D3D_API int d3d_op_linear_ln(d3d_handle* h, const float* a_dev, const float* w_dev, const float* bias_dev,
                     const float* residual_dev, const float* gamma_dev, const float* beta_dev, float eps,
                     float* x_out_dev, float* ln_out_dev, int64_t M, int32_t K, void* stream);

/* The deferred-norm2 pair of the F4C tcgen05 path (MODEL:127-128, 51-52) on explicit operands:
 *   x_out [M,512]    = a . w^T + bias + residual                       (proj: EPI_F32_EMIT, also emits x as an operand)
 *   hid_out [M,1024] = gelu(LayerNorm(x_out; gamma, beta, eps) . w2^T + b2)   (fc1: EPI_GELU_DLN on that operand, with
 *                      w2 folded with gamma at "load time" and the row statistics applied in the epilogue),
 * hid_out read back from the block-scaled operand format it is written in.  K = columns of a, K % 128 == 0. */
D3D_API int d3d_op_linear_dln_linear(d3d_handle* h, const float* a_dev, const float* w_dev, const float* bias_dev,
                             const float* residual_dev, const float* gamma_dev, const float* beta_dev, float eps,
                             const float* w2_dev, const float* b2_dev, float* x_out_dev, float* hid_out_dev, int64_t M,
                             int32_t K, void* stream);

/* Runs one attention core like d3d_op_attention but returns the result in the raw GEMM A-operand format the proj
 * GEMM consumes: hi_out_dev [T, C] fp16 and second_out_dev [T, 2*C] bytes (operand format of the handle's gemm_mode:
 * fp16 lo[C], or uint8 e5m2(x * 2^-8)[C] | e5m2((x - hi) * 2^4)[C]; for the D3D_GEMM_*_F4C modes the buffer holds
 * [T][C] bytes = C e2m1 nibbles of q4(x) | C nibbles of q4(x - hi) per row, followed by [T][C/16] ue8m0 scale bytes per
 * row (k-blocks of 32 elements: 16 of the first part, then 16 of the second), element 2i in the low nibble of byte i). */
D3D_API int d3d_debug_attention_operand(d3d_handle* h, const float* qkv_dev, void* hi_out_dev, void* second_out_dev,
                                int32_t B, int32_t spatial, int32_t attn_mode, void* stream);

/* One row-wise kernel of the hot path in isolation: exactly one launch through the production launcher, on the
 * handle's weights and its own X / A workspace, with the arguments the denoiser call passes.  T = B*F*J rows.
 *   D3D_ROWWISE_LIFT      in_dev x5 [T,5]; out_dev X [T,C] = fusion_layer(x5) + Spatial_pos_embed + time vector of
 *                         block 0; operand = norm1 of block 0 (X)                          (MODEL:250, 230-233, 113-116, 127)
 *   D3D_ROWWISE_POSTNORM  in_dev X [T,C] leaving block `block`-1 (1 <= block < 2*depth); out_dev X entering `block` =
 *                         Spatial_norm (block-1 even) / Temporal_norm (block-1 odd) of X (+ Temporal_pos_embed when
 *                         block == 1) + time vector of `block`; operand = norm1 of `block` (X)  (MODEL:236/245, 239-242)
 *   D3D_ROWWISE_NORM2     in_dev X [T,C]; operand = norm2 of `block` (X), eps 1e-6; out_dev unused (may be NULL)
 *                                                                                                          (MODEL:128)
 *   D3D_ROWWISE_HEAD      in_dev X [T,C] leaving the last block; out_dev [T,3] = head.1(head.0 LN (1e-5) of
 *                         Temporal_norm(X)), the forward_denoise form (MODEL:245, 255-257); no operand
 * Time vectors (LIFT / POSTNORM, handles with with_time_emb): t_dev [B] int64.  shared_t != 0 adds clip 0's vector to
 * every row, as the DDIM loop does (one t per step): with the default D3D_LN_ROWS this selects the two-rows-per-warp
 * kernels, and LIFT reads x5 de-interleaved into the sampler's x2d / y arrays.  shared_t == 0 adds each clip's own
 * vector, as forward_denoise does: one row per warp.  D3D_LN_ROWS=1 selects the one-row kernels throughout.  The
 * operand comes back in the layout of d3d_debug_attention_operand (hi_out_dev [T,C] fp16, second_out_dev [T,2*C]
 * bytes); rows the launch leaves unwritten read back as NaN halves / 0xff bytes. */
enum {
  D3D_ROWWISE_LIFT = 0,
  D3D_ROWWISE_POSTNORM = 1,
  D3D_ROWWISE_NORM2 = 2,
  D3D_ROWWISE_HEAD = 3
};
D3D_API int d3d_debug_rowwise(d3d_handle* h, int32_t op, int32_t block, const float* in_dev, const int64_t* t_dev,
                              int32_t shared_t, int32_t B, float* out_dev, void* hi_out_dev, void* second_out_dev,
                              void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DIFF3D_B200_H_ */
