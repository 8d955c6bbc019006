// Launcher declarations shared by the engine and the kernel translation units.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace d3d {

// The model width C (embed_dim) is a compile-time parameter of every hot-path kernel, instantiated for C = 512 and
// C = 256; a handle picks its instantiation once, from d3d_config::embed_dim.  The head count is the reference's fixed 8,
// so the head dimension is C / 8 (64 or 32) and the MLP hidden width 2 C (mlp_ratio 2).
constexpr int kHeads = 8;
template <int C>
struct Width {
  static_assert(C == 256 || C == 512, "the kernels are instantiated for embed_dim 256 and 512");
  static constexpr int kC = C;
  static constexpr int kHd = C / kHeads;     // head_dim
  static constexpr int kHidden = 2 * C;      // mlp hidden
  static constexpr int kQkvRow = 4 * C;      // halves per token row of the packed q|k|v_hi|v_lo tensor
};
inline bool width_supported(int C) { return C == 256 || C == 512; }

// ------------------------------------------------------------------ GEMM
// EPI_F32        out_f32[M,N] = acc + bias (+ residual)
// EPI_GELU_SPLIT out_hi/out_lo[M,N] = split_fp16(gelu_erf(acc + bias))            (fc1 -> A operand of fc2)
// EPI_QKV16      N == 3 C: out_qkv[M, 4 C] fp16 rows = q(C) | k(C) | v_hi(C) | v_lo(C)
//                (q, k rounded to fp16; v kept as a hi/lo pair so that the GRAND "- V" term stays exact).  The launcher runs
//                the C = 256 rows (N == 768) on the EPI_QKV16_256 instantiation.
// EPI_F32_RED    out_f32[M,N] += acc + bias: the in-place residual update of proj / fc2 (MODEL:127-128) as a TMA REDUCTION
//                (cp.reduce.async.bulk.tensor .add.f32): the L2 adds the staged fp32 chunk to X, so the residual rows
//                never travel L2 -> SM -- the link that bounds all four GEMMs.  Needs the `out` tensor map of GemmMaps
//                ({32 floats x 32 rows} boxes over out_f32); same single fp32 rounding as (acc + bias) + x.
// The values are part of the kernel symbols (gemm_tc_kernel<..., EPI, ...>) that the captures under profiles/ name, so
// EPI_F32_RED keeps 6.
enum GemmEpi { EPI_F32 = 0, EPI_GELU_SPLIT = 1, EPI_QKV16 = 2, EPI_QKV16_256 = 3, EPI_F32_RED = 6 };
// embed_dim of a packed q|k|v_hi|v_lo epilogue
constexpr int qkv_epi_width(int epi) { return epi == EPI_QKV16_256 ? 256 : 512; }

// The GEMM kernels take it as a __grid_constant__ parameter: fields are read from parameter space where they are used.
// Passed as a plain by-value struct of at most 128 bytes, it is loaded into registers at kernel entry instead (ptxas on
// this struct: up to 22 more registers per thread, and spills in the fp32 epilogue kernels).
struct GemmParams {
  int M, N, K;
  const float* bias;      // [N] (never null)
  const float* residual;  // [M,N] or null; may alias out_f32
  float* out_f32;         // EPI_F32
  __half* out_hi;         // EPI_GELU_SPLIT
  __half* out_lo;
  __half* out_qkv;        // EPI_QKV16
  uint8_t* out_sf;        // EPI_GELU_SPLIT with FMT_F4C: scale-factor array of the output operand (K_out = N)
  // L2 policy knobs (defaults chosen from ncu DRAM-traffic measurements, see DESIGN.md): TMA eviction priority of the
  // activation (A) and weight (B) operand loads (0 normal, 1 evict_last, 2 evict_first) and streaming (evict-first)
  // output stores / residual loads
  int hint_a, hint_b, stream_out;
  int n_inner;            // tile order of the persistent tcgen05 kernel: 1 = all n-tiles of an m-tile on the same CTA pair
  int prefetch_a;         // FMT_F4C, n-inner: L2-prefetch the A rows of the unit's next m-tile while the current one runs
};

// A: [M,K] fp16 (hi, lo), W: [N,K] fp16 (hi, lo); K-major.  Tensor maps use a {64, 128} box, SWIZZLE_128B.
struct GemmMaps {
  CUtensorMap a_hi, a_lo, b_hi, b_lo;
  CUtensorMap b_hi64, b_lo64;     // weight maps with 64-row boxes (multicast slices of the pair-cluster kernel)
  CUtensorMap a_sf, b_sf;         // FMT_F4C: scale-factor arrays (make_sf_map)
  CUtensorMap out;                // EPI_F32_RED: fp32 [M, N] destination, {32 x 32} boxes, SWIZZLE_128B (make_f32_tile_map)
};

// passes: 3 (split fp16), 1 (fp16), 2 (FMT_F8C: fp16 main + e5m2 corrections; the *_lo maps are the uint8 c8 maps) or
// 4 (FMT_F4C: fp16 main + block-scaled e2m1 corrections; *_lo = uint8 c4 maps [rows, K bytes], *_sf = scale factors;
// CTA-pair kernel only, N % 256 == 0, K % 128 == 0).
// cta_group 1: one CTA per 128 x bn tile (bn 128 or 256, N % bn == 0);
// cta_group 2: a CTA pair per 256 x 256 tile (tcgen05.mma.cta_group::2, N % 256 == 0, bn ignored).
// pair_cluster 2 (F8C + cta_group 2 only): clusters of two CTA pairs sharing the weight tile through TMA multicast.
// epi_warps 16 (F8C CTA-pair kernel, GELU / QKV epilogues): 16 epilogue warps per CTA instead of 8.
cudaError_t launch_gemm_tc(const GemmMaps& maps, const GemmParams& p, int epi, int passes, int bn, int cta_group,
                           int pair_cluster, int epi_warps, int num_sms, cudaStream_t st);
cudaError_t launch_gemm_simt(const __half* a_hi, const __half* a_lo, const uint8_t* a_sf, const __half* b_hi,
                             const __half* b_lo, const uint8_t* b_sf, const GemmParams& p, int epi, int fmt,
                             cudaStream_t st);
// One-time per-device kernel attribute setup (dynamic shared memory opt-in); call outside graph capture.
cudaError_t configure_gemm_tc();
cudaError_t configure_attention();
cudaError_t configure_attention_mma();
// Build a K-major fp16 operand map for a [rows, K] row-major matrix / a uint8 map for a [rows, row_bytes] c8 array.
int make_operand_map(CUtensorMap* out, const __half* base, int64_t rows, int64_t K, int box_rows = 128);
int make_operand_map_u8(CUtensorMap* out, const void* base, int64_t rows, int64_t row_bytes, int box_rows = 128);
int make_sf_map(CUtensorMap* out, const void* base, int64_t total_bytes);
// fp32 [rows, N] row-major matrix, {32 floats x 32 rows} boxes, SWIZZLE_128B (the epilogue's staging-buffer layout)
int make_f32_tile_map(CUtensorMap* out, const float* base, int64_t rows, int N);

// ------------------------------------------------------------------ row-wise (one warp per C-wide token row)
// The row-wise and attention launchers take the handle's width C (256 or 512) and run that instantiation.
struct LnParams {
  const float* gamma;
  const float* beta;
};

// fp32 [rows, K] -> GEMM operand arrays (hi + second, see operand.cuh; fmt = OperandFmt; weights at load time,
// op-level tests) and back (activation operands only).
// absmax (optional, device float[2], zeroed by the caller): [0] = max |x| over the finite inputs, [1] = 1 if any input
// was NaN / Inf -- the load-time range guard of d3d_load_weights.
// sf: the operand's scale-factor array (FMT_F4C only, else ignored / null).
cudaError_t launch_split(const float* in, __half* hi, __half* second, uint8_t* sf, int64_t rows, int K, int fmt,
                         int is_weight, cudaStream_t st, float* absmax = nullptr);
cudaError_t launch_merge(const __half* hi, const __half* second, const uint8_t* sf, float* out, int64_t rows, int K,
                         int fmt, cudaStream_t st);

// FMT_F4C scale factors of `rows` rows in atom layout -> row-major [rows][K / 16] bytes (test read-back)
cudaError_t launch_sf_rows(const uint8_t* sf, uint8_t* out, int64_t rows, int K, cudaStream_t st);

// X = [x2d,y] . Wf^T + bf + spos[j] (+ tvec[sample]);  A = LN(X; ln1)  (MODEL:250, 230-233, 113-116, 127)
cudaError_t launch_lift_ln(int C, const float* x2d, const float* y, const float* x5, const float* wf_t /*[5][C]*/,
                           const float* bf, const float* spos /*[J][C]*/, const float* tvec, int64_t tvec_stride,
                           LnParams ln1, float* X, __half* a_hi, __half* a_lo, uint8_t* a_sf, int fmt, int64_t T, int J,
                           int tokens_per_clip, cudaStream_t st);
// X = LN(X; post) (+ tpos[f]) (+ tvec[sample]);  A = LN(X; ln1)   (MODEL:236/245, 239-242, 113-116, 127)
cudaError_t launch_postnorm_add_ln(int C, float* X, LnParams post, const float* tpos /*[F][C] or null*/,
                                   const float* tvec, int64_t tvec_stride, LnParams ln1, __half* a_hi,
                                   __half* a_lo, uint8_t* a_sf, int fmt, int64_t T, int J, int F, cudaStream_t st);
// A = LN(X; ln)  (MODEL:128 norm2)
cudaError_t launch_ln_split(int C, const float* X, LnParams ln, float eps, __half* a_hi, __half* a_lo, uint8_t* a_sf, int fmt,
                            int64_t T, cudaStream_t st);
// out = LN(x) fp32, the per-row arithmetic of the kernels above (d3d_op_layernorm: reference of their operands)
cudaError_t launch_ln_f32(int C, const float* x, LnParams ln, float eps, float* out, int64_t T, cudaStream_t st);

struct DdimStep {      // DIFF:287-297 scalars; last != 0 -> y_next = x0 (DIFF:283-285)
  float sqrt_alpha_next, c, alpha, sqrt_one_minus, sigma;
  int last, clip;
};
// x0 = head(LN(LN(X; post, 1e-6); head.0, 1e-5)); clamp; DDIM update.  (MODEL:245,255; DIFF:256,287-297)
// If out3 != null only x0 is written there (forward_denoise); else y is updated in place.
cudaError_t launch_head_ddim(int C, const float* X, LnParams post, LnParams head_ln, const float* wh /*[3][C]*/,
                             const float* bh, DdimStep s, float* y, const float* noise, float* out3,
                             float* trace_y, float* trace_x0, int trace_stride, int trace_idx, int64_t T,
                             cudaStream_t st);

cudaError_t launch_tta_merge(const float* y, const float* yf, const int32_t* perm /*[J] device*/, float scale,
                             float* out, int64_t n_frames, int J, cudaStream_t st);
cudaError_t launch_mpjpe(const float* pred, const float* gt, const uint8_t* mask, int64_t n_frames, int J,
                         double* acc, cudaStream_t st);

// Protocol #1/#2/#3 + velocity sums (metrics.cu): acc[6] fp64 = sum mpjpe, sum n_mpjpe, sum p_mpjpe, joints, sum vel, vel joints
// vel_tmp: device double[2] scratch owned by the handle (per-call velocity sum / count before the reference's weighting)
cudaError_t launch_pose_metrics(const float* pred, const float* gt, const int64_t* sel /*or null*/, int64_t n_sel, int J,
                                double* acc, double* vel_tmp, cudaStream_t st);

// Grouped per-joint histogram of joint errors (metrics.cu, d3d_pck_accumulate): counts[g][j][k] += listed frames of group
// g whose joint-j error is < thr.t[k], err_sum[g][j] += those errors, frames[g] += listed frames of group g.
constexpr int kPckMaxThresholds = 64;
constexpr int kPckMaxGroups = 65536;
constexpr int kPckSmemBinBytes = 32 * 1024;   // histograms up to this size are built in shared memory per block
struct PckThresholds {                        // passed by value: no device copy, graph-capturable
  float t[kPckMaxThresholds];                 // t[0] < t[1] < ... < t[n-1], finite (checked by the caller)
  int n;
};
cudaError_t launch_pck_hist(const float* pred, const float* gt, const int64_t* sel /*or null*/,
                            const int32_t* group /*[n_frames] or null*/, int64_t n_sel, int J, const PckThresholds& thr,
                            int n_groups, int64_t* counts, double* err_sum, int64_t* frames, int num_sms,
                            cudaStream_t st);

// ------------------------------------------------------------------ windowing (packed sequences <-> F-frame windows)
cudaError_t launch_window_gather(const float* seq2d, const int64_t* start, const int32_t* perm /*[J] device*/, float* x2d,
                                 float* x2d_flip /*or null*/, int64_t n_win, int F, int J, cudaStream_t st);
cudaError_t launch_window_scatter(const float* pred, const int64_t* start, const int32_t* first_valid, float* seq3d,
                                  int64_t n_win, int F, int J, cudaStream_t st);

// ------------------------------------------------------------------ attention
// qkv: packed fp16 [T, 4 C] rows q | k | v_hi | v_lo (EPI_QKV16).  Output [T, C]: GEMM A operand (o_hi + second
// array in format fmt, operand.cuh) or fp32.  The mma.sync and CUDA-core kernels below (validation modes) are built for
// C = 512 only; the tcgen05 kernel for both widths.
cudaError_t launch_attn_spatial(const __half* qkv, __half* o_hi, __half* o_lo, float* o_f32, int fmt, int64_t n_groups,
                                int J, cudaStream_t st);
cudaError_t launch_attn_temporal_mma(const __half* qkv, __half* o_hi, __half* o_lo, float* o_f32, int fmt, int B, int F,
                                     int J, cudaStream_t st);
// tcgen05 / TMEM / TMA temporal kernel (attention_tc.cu), 1 <= F <= 256 (F <= 64: 2 or 4 joints packed per tile).  Its tensor maps are bound to one packed
// qkv array and one output operand (hi + second array in format fmt) of up to max_clips clips.
struct AttnTcMaps {
  CUtensorMap qkv, o_hi, o_second;
  CUtensorMap o_hi_tail, o_second_tail;   // spatial mode: store boxes of the last (shorter) frame group of a clip
};
int make_attn_tc_maps(int C, AttnTcMaps* maps, const __half* qkv, __half* o_hi, __half* o_second, int fmt, int F, int J,
                      int64_t max_clips);
// spatial mode of the same kernel (J == 17): units of (clip, 7 frames = 119 consecutive tokens, head), block-diagonal mask
int make_attn_tc_maps_spatial(int C, AttnTcMaps* maps, const __half* qkv, __half* o_hi, __half* o_second, int fmt, int64_t tokens,
                              int F);
// o_sf: scale-factor array of the output operand (FMT_F4C; null otherwise)
cudaError_t launch_attn_spatial_tc(int C, const AttnTcMaps& maps, uint8_t* o_sf, int fmt, int B, int F, int num_sms, cudaStream_t st);
cudaError_t configure_attention_tc();
// wg2 != 0 (FMT_F4C, F > 64, C = 512): two softmax warpgroups per 128-query slot (attn_temporal_tc2_kernel)
cudaError_t launch_attn_temporal_tc(int C, const AttnTcMaps& maps, const __half* qkv, uint8_t* o_sf, int fmt, int B, int F, int J,
                                    int num_sms, cudaStream_t st, int wg2 = 0);
// CUDA-core validation kernels (fp32 arithmetic on the same packed input)
cudaError_t launch_attn_temporal_simt(const __half* qkv, __half* o_hi, __half* o_lo, float* o_f32, int fmt, int B, int F,
                                      int J, cudaStream_t st);
cudaError_t launch_attn_generic_simt(const __half* qkv, __half* o_hi, __half* o_lo, float* o_f32, int fmt, int n_seq,
                                     int N, int64_t seq_stride_tokens_outer, int inner, int64_t tok_stride,
                                     cudaStream_t st);
// fp32 [T, 3 C] -> packed fp16 [T, 4 C] (op-level test entry point)
cudaError_t launch_pack_qkv16(int C, const float* qkv_f32, __half* out, int64_t T, cudaStream_t st);

// ------------------------------------------------------------------ time embedding
// out[r] = float(t[r]): the per-sample timesteps of forward_denoise stay on the device (no host round trip)
cudaError_t launch_t_to_f32(const int64_t* t, int R, float* out, cudaStream_t st);
// e[r, 0:C/2] = sin(t_r * f_i), e[r, C/2:C] = cos(t_r * f_i)   (MODEL:29-36)
cudaError_t launch_sincos(int C, const float* t, int R, float* out, cudaStream_t st);
// out[r, n] = act_in(in[r, :]) . W[n, :] + b[n];  act_in: 0 none, 1 gelu(erf), 2 silu.  out row stride given.
cudaError_t launch_small_linear(const float* in, int R, int K, const float* W, const float* b, int N, int act_in,
                                float* out, int64_t out_row_stride, cudaStream_t st);

}  // namespace d3d
