// Host side of libdiff3d_b200.so: handle, weight packing, workspace, kernel sequencing of one denoiser call
// (MODEL:249-257), the S-step DDIM loop (DIFF:263-300) with CUDA-graph replay, and the extern "C" boundary
// declared in include/diff3d_b200.h.
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/diff3d_b200.h"
#include "kernels.cuh"
#include "operand.cuh"

using namespace d3d;

namespace {

// message of the calling thread's last failed d3d_create: handles may be created from several threads at once
thread_local std::string g_create_error;

struct Lin {
  int N = 0, K = 0;
  __half* hi = nullptr;
  __half* lo = nullptr;
  uint8_t* sf = nullptr;        // FMT_F4C: scale factors, behind the c4 bytes inside the `lo` allocation
  float* bias = nullptr;
  bool have_w = false;
  CUtensorMap m_hi, m_lo, m_sf;
  CUtensorMap m_hi64, m_lo64;   // 64-row boxes (pair-cluster multicast slices)
};

struct Blk {
  float *n1g = nullptr, *n1b = nullptr, *n2g = nullptr, *n2b = nullptr;
  Lin qkv, proj, fc1, fc2;
  float *tw = nullptr, *tb = nullptr;   // per-block time Linear(1024 -> 512), fp32
  bool have_t = false;
  // deferred norm2 (d3d_handle::defer_ln2): the raw fc1 weight stays on the device so that it can be re-folded with
  // norm2.weight whenever either is (re)loaded; fc1_s = column sums of the folded weight, fc1_c = folded bias
  float *fc1_raw = nullptr, *fc1_s = nullptr, *fc1_c = nullptr;
  bool fold_dirty = false;
};

struct OperandBuf {   // a GEMM A operand living in the workspace
  __half* hi = nullptr;
  __half* lo = nullptr;
  uint8_t* sf = nullptr;        // FMT_F4C: scale factors, behind the c4 bytes inside the `lo` allocation
  CUtensorMap m_hi, m_lo, m_sf;
};

}  // namespace

struct d3d_handle {
  d3d_config cfg{};
  int F = 0, J = 0, nblk = 0, num_sms = 148;
  int fmt = FMT_SPLIT16;   // GEMM operand format of the workspace and the packed weights (operand.cuh)
  int64_t tok_cap = 0;   // workspace rows (multiple of 128)
  std::string err;
  int64_t launches = 0;

  // parameters
  std::vector<Blk> blk;
  float *wf_t = nullptr, *bf = nullptr, *spos = nullptr, *tpos = nullptr;
  float *sn_g = nullptr, *sn_b = nullptr, *tn_g = nullptr, *tn_b = nullptr;
  float *hg = nullptr, *hb = nullptr, *wh = nullptr, *bh = nullptr;
  float *tm1w = nullptr, *tm1b = nullptr, *tm3w = nullptr, *tm3b = nullptr;
  std::map<std::string, bool> loaded;

  // workspace
  float* X = nullptr;
  __half* QKV = nullptr;     // packed fp16 q | k | v_hi | v_lo, [tok_cap, 2048]
  OperandBuf A, ATT, H;
  // Deferred norm2 (FMT_F4C tcgen05 path): the proj epilogue emits x itself as fc1's A operand plus per-row partial sums
  // (EPI_F32_EMIT), the fc1 epilogue applies the LayerNorm (EPI_GELU_DLN); no ln_split pass (DESIGN.md 4.1)
  bool defer_ln2 = false;
  float2* ln_stats = nullptr;   // [8][tok_cap] (sum, sum of squares) per 64 columns
  CUtensorMap m_x;              // fp32 [tok_cap, 512] view of X in {32 x 32} boxes: destination of the EPI_F32_RED epilogue
  bool have_m_x = false;
  AttnTcMaps attn_tc;        // tcgen05 temporal attention: maps bound to QKV -> ATT
  bool have_attn_tc = false;
  AttnTcMaps attn_sp;        // spatial mode of the same kernel (J == 17)
  bool have_attn_sp = false;
  float *in_x2d = nullptr, *y = nullptr, *in_noise = nullptr;
  int64_t in_noise_cap = 0;
  float *t_f32 = nullptr, *e0 = nullptr, *h1 = nullptr, *h2 = nullptr;   // time-MLP scratch, max(max_clips, S) rows
  int t_rows_cap = 0;
  float* tv_steps = nullptr;     // [S, nblk, 512] table for the DDIM loop
  int tv_cap = 0;
  float* tv_general = nullptr;   // [max_clips, nblk, 512] for per-sample t
  int32_t* perm_dev = nullptr;
  int32_t perm_host[64];
  bool perm_valid = false;

  // schedule
  int S = 0;
  std::vector<int> times;
  std::vector<DdimStep> steps;
  bool have_schedule = false, table_valid = false, need_noise = false;

  // per-kernel-class device timing (d3d_profile_*): events bracket every launch of the un-graphed sampler
  bool prof = false;
  std::vector<cudaEvent_t> prof_pool;
  struct ProfRec { int cls; cudaEvent_t a, b; };
  std::vector<ProfRec> prof_recs;
  size_t prof_next = 0;

  std::map<int, cudaGraphExec_t> graphs;
  std::map<int, int64_t> graph_launches;
  cudaStream_t cap_stream = nullptr;
  cudaEvent_t table_event = nullptr;   // recorded after the time table of the current schedule was computed
  int64_t qkv_rows_dirty = 0;          // high-water mark of token rows ever written into QKV (see prep_batch)
  float* absmax_dev = nullptr;         // load-time |w| maximum of the last split weight (range guard)
  double* vel_tmp = nullptr;           // per-call (sum, count) of the velocity error (d3d_pose_metrics_accumulate)
  std::vector<void*> allocs;
  int64_t alloc_bytes = 0;             // device bytes owned by the handle (d3d_workspace_bytes)
};

namespace {

#define CK(expr)                                                                                       \
  do {                                                                                                 \
    cudaError_t _e = (expr);                                                                           \
    if (_e != cudaSuccess) {                                                                           \
      char _b[512];                                                                                    \
      snprintf(_b, sizeof(_b), "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      h->err = _b;                                                                                     \
      return static_cast<int>(_e);                                                                     \
    }                                                                                                  \
  } while (0)
// kernel launch: counted
#define KL(expr)       \
  do {                 \
    CK(expr);          \
    ++h->launches;     \
  } while (0)

// kernel launch of class `cls` (D3D_PROF_*): counted, and bracketed by events when profiling is on
#define KLP(cls, st, expr)                                          \
  do {                                                              \
    cudaEvent_t _a = nullptr, _b = nullptr;                         \
    if (h->prof) {                                                  \
      _a = prof_event(h);                                           \
      _b = prof_event(h);                                           \
      if (_a && _b) CK(cudaEventRecord(_a, st));                    \
    }                                                               \
    KL(expr);                                                       \
    if (h->prof && _a && _b) {                                      \
      CK(cudaEventRecord(_b, st));                                  \
      h->prof_recs.push_back(d3d_handle::ProfRec{cls, _a, _b});     \
    }                                                               \
  } while (0)

cudaEvent_t prof_event(d3d_handle* h) {
  if (h->prof_next == h->prof_pool.size()) {
    cudaEvent_t e = nullptr;
    if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
    h->prof_pool.push_back(e);
  }
  return h->prof_pool[h->prof_next++];
}

int fail(d3d_handle* h, int code, const std::string& msg) {
  h->err = msg;
  return code;
}

template <typename T>
int dev_alloc(d3d_handle* h, T** p, int64_t n, bool zero = true) {
  void* q = nullptr;
  CK(cudaMalloc(&q, static_cast<size_t>(n) * sizeof(T)));
  if (zero) CK(cudaMemset(q, 0, static_cast<size_t>(n) * sizeof(T)));
  h->allocs.push_back(q);
  h->alloc_bytes += static_cast<int64_t>(n) * static_cast<int64_t>(sizeof(T));
  *p = static_cast<T*>(q);
  return 0;
}

#ifndef D3D_ATTN_TC_F4C
#define D3D_ATTN_TC_F4C 1     // 0: route FMT_F4C attention through the mma.sync kernels + a split pass (bring-up A/B)
#endif

// fp16 main operand: finite up to 65504; the e5m2 images (w 2^-4, (w - hi) 2^8 <= |w| / 8) stay below e5m2's 57344
constexpr float kMaxWeightAbs = 65504.0f;

int mode_fmt(int gemm_mode) {
  if (gemm_mode == D3D_GEMM_TC_F4C || gemm_mode == D3D_GEMM_SIMT_F4C) return FMT_F4C;
  return (gemm_mode == D3D_GEMM_TC_F8C || gemm_mode == D3D_GEMM_SIMT_F8C) ? FMT_F8C : FMT_SPLIT16;
}

// tensor maps of an operand: fp16 hi [rows,K]; second array = fp16 lo [rows,K] or uint8 c8 [rows,2K]
int make_maps(CUtensorMap* m_hi, CUtensorMap* m_second, const __half* hi, const __half* second, int64_t rows, int K,
              int fmt, int box_rows = 128) {
  if (make_operand_map(m_hi, hi, rows, K, box_rows)) return -1;
  if (fmt == FMT_F8C) return make_operand_map_u8(m_second, second, rows, 2 * static_cast<int64_t>(K), box_rows);
  if (fmt == FMT_F4C) return make_operand_map_u8(m_second, second, rows, K, box_rows);      // c4: K bytes per row
  return make_operand_map(m_second, second, rows, K, box_rows);
}
// FMT_F4C: the scale-factor array sits behind the c4 bytes of the second array (2 K bytes per row were allocated, c4
// takes K and the scales K / 16); rows must be a multiple of 128 (whole scale-factor atoms)
int make_sf(uint8_t** sf, CUtensorMap* m_sf, __half* second, int64_t rows, int K, int fmt) {
  *sf = nullptr;
  if (fmt != FMT_F4C) return 0;
  if (rows % 128 != 0 || K % 64 != 0) return -1;
  *sf = reinterpret_cast<uint8_t*>(second) + op_sf_base(rows, K);
  return make_sf_map(m_sf, *sf, rows * (K / 16));
}

int alloc_operand(d3d_handle* h, OperandBuf* o, int64_t rows, int K) {
  int r;
  if ((r = dev_alloc(h, &o->hi, rows * K))) return r;
  if ((r = dev_alloc(h, &o->lo, rows * K))) return r;
  if (make_maps(&o->m_hi, &o->m_lo, o->hi, o->lo, rows, K, h->fmt) || make_sf(&o->sf, &o->m_sf, o->lo, rows, K, h->fmt))
    return fail(h, -20, "cuTensorMapEncodeTiled failed for a workspace operand");
  return 0;
}

int alloc_lin(d3d_handle* h, Lin* l, int N, int K) {
  l->N = N;
  l->K = K;
  int r;
  if ((r = dev_alloc(h, &l->hi, static_cast<int64_t>(N) * K))) return r;
  if ((r = dev_alloc(h, &l->lo, static_cast<int64_t>(N) * K))) return r;
  if ((r = dev_alloc(h, &l->bias, N))) return r;
  if (make_maps(&l->m_hi, &l->m_lo, l->hi, l->lo, N, K, h->fmt) ||
      make_maps(&l->m_hi64, &l->m_lo64, l->hi, l->lo, N, K, h->fmt, 64) || make_sf(&l->sf, &l->m_sf, l->lo, N, K, h->fmt))
    return fail(h, -20, "cuTensorMapEncodeTiled failed for a weight operand");
  return 0;
}

int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v && *v ? atoi(v) : dflt;
}

int pick_cg(int N) {
  const int cg = env_int("D3D_GEMM_CG", 2);
  return (cg == 2 && N % 256 == 0) ? 2 : 1;
}

// pairs per cluster of the F8C CTA-pair kernel: 2 = weight-tile TMA multicast across two pairs, 1 = none (default:
// measured on B200 the multicast variant is ~3 % SLOWER, profiles/r01f_micro.log -- L2 already serves the identical
// unicast requests of neighbouring pairs, and 4-CTA clusters leave SMs of 18-SM GPCs idle)
int pick_cs(int64_t M) {
  const int cs = env_int("D3D_GEMM_CS", 1);
  return (cs == 2 && M > 256) ? 2 : 1;
}

int pick_bn(const d3d_handle* h, int64_t M, int N) {
  int bn = env_int("D3D_GEMM_BN", 0);
  if (bn == 128 || bn == 256) return (N % bn == 0) ? bn : 128;
  if (N % 256 != 0) return 128;
  const int64_t tiles256 = ((M + 127) / 128) * (N / 256);
  return tiles256 >= 2 * h->num_sms ? 256 : 128;
}

struct LnFuse {           // LayerNorm fused behind an EPI_F32 GEMM (EPI_F32_LN): parameters and destination operand
  const float* gamma;
  const float* beta;
  float eps;
  OperandBuf* dst;
};

// proj + norm2 in one kernel: CTA-pair F8C tcgen05 GEMM with the n-inner tile order only
bool can_fuse_ln(const d3d_handle* h, int mode) {
  return mode == D3D_GEMM_TC_F8C && h->fmt == FMT_F8C && pick_cg(kC) == 2 && env_int("D3D_GEMM_N_INNER", 1) == 1;
}
// OFF by default.  Measured on B200 at cfg3 (profiles/r01s_bench_fuse*.json): correct, but SLOWER -- GEMM class
// 2727 -> 3069 ms per step for 198 ms of LayerNorm kernels saved (3802 -> 3943 ms per step).  Between its two passes
// the epilogue holds BOTH accumulators, so its residual loads / operand stores are no longer hidden behind the next
// tile's mainloop (~15 us per 128 x 256 pass with 8 warps, against 17 us of mainloop per row tile).
bool fuse_ln_enabled() { return env_int("D3D_GEMM_FUSE_LN", 0) == 1; }

struct DeferLn {          // deferred LayerNorm (EPI_F32_EMIT producer / EPI_GELU_DLN consumer)
  const OperandBuf* emit; // EPI_F32_EMIT: destination operand of x
  float2* stats;
  const float* colsum;    // EPI_GELU_DLN
  const float* cbias;     // EPI_GELU_DLN: folded bias (replaces the Linear's own)
  float eps;
};

// out = epilogue(Aop . W^T + bias)
int run_gemm(d3d_handle* h, const OperandBuf& a, const Lin& w, int64_t M, int epi, const float* residual,
             float* out_f32, __half* out_hi, __half* out_lo, __half* out_qkv, int mode, cudaStream_t st,
             const LnFuse* ln = nullptr, uint8_t* out_sf = nullptr, const DeferLn* dl = nullptr,
             const CUtensorMap* out_map = nullptr) {
  GemmParams p{};
  // in-place residual update on the F4C tcgen05 kernel: let the L2 do the add (TMA reduction) instead of pulling the
  // residual rows into the SM (D3D_GEMM_RED=0: the load-add-store epilogue)
  if (epi == EPI_F32 && !ln && out_map && residual && residual == out_f32 && mode == D3D_GEMM_TC_F4C && pick_cg(w.N) == 2 &&
      env_int("D3D_GEMM_RED", 1) == 1)
    epi = EPI_F32_RED;
  p.out_sf = out_sf;
  if (dl) {
    if (mode != D3D_GEMM_TC_F4C) return fail(h, -3, "the deferred-LayerNorm epilogues need the F4C tcgen05 GEMM");
    p.ln_stats = dl->stats;
    p.ln_eps = dl->eps;
    if (epi == EPI_F32_EMIT) {
      p.emit_hi = dl->emit->hi; p.emit_c4 = reinterpret_cast<uint8_t*>(dl->emit->lo); p.emit_sf = dl->emit->sf;
    } else {
      p.ln_colsum = dl->colsum;
    }
  }
  if (ln) {
    epi = EPI_F32_LN;
    p.ln_gamma = ln->gamma; p.ln_beta = ln->beta; p.ln_eps = ln->eps;
    p.ln_hi = ln->dst->hi; p.ln_second = ln->dst->lo;
  }
  p.M = static_cast<int>(M);
  p.N = w.N;
  p.K = w.K;
  p.bias = (dl && epi == EPI_GELU_DLN) ? dl->cbias : w.bias;
  p.residual = residual;
  p.out_f32 = out_f32;
  p.out_hi = out_hi;
  p.out_lo = out_lo;
  p.out_qkv = out_qkv;
  // measured (profiles/r01i_hint_sweep.log): evict_last operands + streaming outputs is ~2 % faster than no hints,
  // evict_first activations ~3 % slower (the A tile is re-read by the other n-tiles' CTA pairs out of L2)
  p.hint_a = env_int("D3D_GEMM_HINT_A", 1);
  p.hint_b = env_int("D3D_GEMM_HINT_B", 1);
  p.stream_out = env_int("D3D_GEMM_STREAM_OUT", 1);
  // measured (profiles/r01q_*): DRAM reads of the qkv GEMM 2.9x -> 1.1x its algorithmic bytes, step time -1.7 %
  p.n_inner = env_int("D3D_GEMM_N_INNER", 1);
  // OFF: measured SLOWER at both distances -- 1 = a whole m-tile ahead (profiles/r02t_gemm_pf.log: qkv +8 %, fc2 +29 %, step
  // 3184 -> 3420 ms), 2 = during the last n-tile of the current m-tile (r02u: qkv +3 %, fc2 +20 %): the prefetch requests
  // ride the same saturated TMA / L2 path as the operand loads they are meant to help
  p.prefetch_a = env_int("D3D_GEMM_PREFETCH_A", 0);
  if (mode == D3D_GEMM_SIMT_FP32 || mode == D3D_GEMM_SIMT_F8C || mode == D3D_GEMM_SIMT_F4C) {
    KLP(D3D_PROF_GEMM, st, launch_gemm_simt(a.hi, a.lo, a.sf, w.hi, w.lo, w.sf, p, epi, mode_fmt(mode), st));
  } else {
    GemmMaps m;
    m.a_hi = a.m_hi; m.a_lo = a.m_lo; m.b_hi = w.m_hi; m.b_lo = w.m_lo;
    m.b_hi64 = w.m_hi64; m.b_lo64 = w.m_lo64;
    m.a_sf = a.m_sf; m.b_sf = w.m_sf;
    if (epi == EPI_F32_RED) m.out = *out_map;
    const int passes = mode == D3D_GEMM_TC_FP16 ? 1 : (mode == D3D_GEMM_TC_F8C ? 2 : (mode == D3D_GEMM_TC_F4C ? 4 : 3));
    // epilogue warps per CTA: 16 pays where the epilogue, not the mainloop, sets the tile time
    // GELU epilogue: 16 warps.  After the epilogue diet 8 warps (one more ring stage) are 2 % faster on the isolated fc1
    // launch (r02r) but 1 % slower in the step (r02s: GEMM class 2157 vs 2139 ms on one box)
    const int ew = (epi == EPI_GELU_SPLIT || epi == EPI_GELU_DLN) ? env_int("D3D_GEMM_EW_GELU", 16)
                 : epi == EPI_QKV16    ? env_int("D3D_GEMM_EW_QKV", 8)
                 : epi == EPI_F32_EMIT ? env_int("D3D_GEMM_EW_EMIT", 8)
                 : epi == EPI_F32_RED  ? 8
                                        : env_int("D3D_GEMM_EW_F32", 8);
    // D3D_GEMM_SMS: run the persistent GEMM on fewer SMs (diagnostic: is the operand feed limited per SM or chip-wide?)
    const int sms = env_int("D3D_GEMM_SMS", h->num_sms);
    KLP(D3D_PROF_GEMM, st, launch_gemm_tc(m, p, epi, passes, pick_bn(h, M, w.N), pick_cg(w.N), pick_cs(M), ew,
                                           sms > 0 && sms < h->num_sms ? sms : h->num_sms, st));
  }
  return 0;
}

bool attn_tc_has_f4c() { return D3D_ATTN_TC_F4C != 0; }

int run_attention(d3d_handle* h, const __half* qkv, __half* o_hi, __half* o_lo, float* o_f32, int B, bool spatial,
                  int mode, cudaStream_t st) {
  const int64_t T_all = static_cast<int64_t>(B) * h->F * h->J;
  const bool tc_path = mode == D3D_ATTN_DEFAULT && qkv == h->QKV &&
                       (spatial ? (h->have_attn_sp && h->J == 17 && env_int("D3D_ATTN_TC_SPATIAL", 1))
                                : (h->have_attn_tc && env_int("D3D_ATTN_TC", 1)));
  if (h->fmt == FMT_F4C && !o_f32 && !(tc_path && attn_tc_has_f4c())) {
    // the mma.sync / CUDA-core attention kernels do not write the block-scaled operand: fp32 result into the (dead)
    // H operand's memory, then one split pass into ATT
    if (o_hi != h->ATT.hi || o_lo != h->ATT.lo) return fail(h, -2, "attention output must be the ATT operand");
    float* scratch = reinterpret_cast<float*>(h->H.hi);
    int r = run_attention(h, qkv, nullptr, nullptr, scratch, B, spatial, mode == D3D_ATTN_DEFAULT ? D3D_ATTN_MMA_SYNC : mode, st);
    if (r) return r;
    KLP(spatial ? D3D_PROF_ATTN_SPATIAL : D3D_PROF_ATTN_TEMPORAL, st,
        launch_split(scratch, h->ATT.hi, h->ATT.lo, h->ATT.sf, T_all, kC, FMT_F4C, 0, st));
    return 0;
  }
  if (spatial) {
    if (mode == D3D_ATTN_SIMT || h->J != 17) {
      KLP(D3D_PROF_ATTN_SPATIAL, st, launch_attn_generic_simt(qkv, o_hi, o_lo, o_f32, h->fmt, B * h->F, h->J, h->J, 1, 1, st));
    } else if (tc_path && (h->fmt != FMT_F4C || attn_tc_has_f4c())) {
      if (!o_f32 && (o_hi != h->ATT.hi || o_lo != h->ATT.lo)) return fail(h, -2, "attention output must be the ATT operand");
      const int64_t T = static_cast<int64_t>(B) * h->F * h->J;
      KLP(D3D_PROF_ATTN_SPATIAL, st, launch_attn_spatial_tc(h->attn_sp, h->ATT.sf, h->fmt, B, h->F, h->num_sms, st));
      if (o_f32) KL(launch_merge(h->ATT.hi, h->ATT.lo, h->ATT.sf, o_f32, T, kC, h->fmt, st));
    } else {
      KLP(D3D_PROF_ATTN_SPATIAL, st, launch_attn_spatial(qkv, o_hi, o_lo, o_f32, h->fmt, static_cast<int64_t>(B) * h->F, h->J, st));
    }
  } else {
    if (mode == D3D_ATTN_SIMT) {
      KLP(D3D_PROF_ATTN_TEMPORAL, st, launch_attn_temporal_simt(qkv, o_hi, o_lo, o_f32, h->fmt, B, h->F, h->J, st));
    } else if (tc_path && (h->fmt != FMT_F4C || attn_tc_has_f4c())) {
      // the tcgen05 kernel's tensor maps are bound to QKV -> ATT; an fp32 result (op-level entry point) is merged
      // from the operand pair afterwards
      if (!o_f32 && (o_hi != h->ATT.hi || o_lo != h->ATT.lo)) return fail(h, -2, "attention output must be the ATT operand");
      KLP(D3D_PROF_ATTN_TEMPORAL, st, launch_attn_temporal_tc(h->attn_tc, qkv, h->ATT.sf, h->fmt, B, h->F, h->J, h->num_sms, st,
                                                              env_int("D3D_ATTN_WG2", 0)));
      if (o_f32) KL(launch_merge(h->ATT.hi, h->ATT.lo, h->ATT.sf, o_f32, static_cast<int64_t>(B) * h->F * h->J, kC, h->fmt, st));
    } else {
      KLP(D3D_PROF_ATTN_TEMPORAL, st, launch_attn_temporal_mma(qkv, o_hi, o_lo, o_f32, h->fmt, B, h->F, h->J, st));
    }
  }
  return 0;
}

int check_weights(d3d_handle* h) {
  static const char* const per_blk[] = {"norm1.weight", "norm1.bias", "attn.qkv.weight", "attn.proj.weight",
                                        "attn.proj.bias", "norm2.weight", "norm2.bias", "mlp.fc1.weight", "mlp.fc1.bias",
                                        "mlp.fc2.weight", "mlp.fc2.bias"};
  std::vector<std::string> need = {"fusion_layer.weight", "fusion_layer.bias", "Spatial_pos_embed", "Temporal_pos_embed",
                                   "Spatial_norm.weight", "Spatial_norm.bias", "Temporal_norm.weight", "Temporal_norm.bias",
                                   "head.0.weight", "head.0.bias", "head.1.weight", "head.1.bias"};
  if (h->cfg.with_time_emb) {
    need.insert(need.end(), {"time_mlp.1.weight", "time_mlp.1.bias", "time_mlp.3.weight", "time_mlp.3.bias"});
  }
  for (int i = 0; i < h->cfg.depth; ++i)
    for (const char* kind : {"STEblocks.", "TTEblocks."}) {
      for (const char* s : per_blk) need.push_back(std::string(kind) + std::to_string(i) + "." + s);
      if (h->cfg.with_time_emb) {
        need.push_back(std::string(kind) + std::to_string(i) + ".time_mlp.1.weight");
        need.push_back(std::string(kind) + std::to_string(i) + ".time_mlp.1.bias");
      }
    }
  for (auto& n : need)
    if (!h->loaded.count(n)) return fail(h, -30, "weights not loaded: missing tensor '" + n + "'");
  for (auto& b : h->blk)
    if (b.fold_dirty) return fail(h, -30, "internal: norm2 / fc1 of a block were not folded");
  return 0;
}

// [R] fp32 timesteps (device) -> table [R, nblk, 512]
int compute_time_table(d3d_handle* h, const float* t_dev, int R, float* table, cudaStream_t st) {
  KL(launch_sincos(t_dev, R, h->e0, st));
  KL(launch_small_linear(h->e0, R, kC, h->tm1w, h->tm1b, 2 * kC, 0, h->h1, 2 * kC, st));
  KL(launch_small_linear(h->h1, R, 2 * kC, h->tm3w, h->tm3b, 2 * kC, 1, h->h2, 2 * kC, st));
  for (int b = 0; b < h->nblk; ++b)
    KL(launch_small_linear(h->h2, R, 2 * kC, h->blk[b].tw, h->blk[b].tb, kC, 2, table + b * kC,
                           static_cast<int64_t>(h->nblk) * kC, st));
  return 0;
}

// The row-wise launches of a denoiser call with the parameters they read (shared by run_blocks and d3d_debug_rowwise).
// tv: time table of the call ([rows][nblk][512], block 0 first) or null; tv_stride: its row stride (0 = one row for
// every clip).
// lift: X = fusion_layer(input) + Spatial_pos_embed + time vector of block 0;  A = norm1 of block 0 (X)
int lift_launch(d3d_handle* h, const float* x2d, const float* y, const float* x5, const float* tv, int64_t tv_stride,
                int64_t T, cudaStream_t st) {
  KLP(D3D_PROF_LIFT, st, launch_lift_ln(x2d, y, x5, h->wf_t, h->bf, h->spos, tv, tv_stride,
                                        LnParams{h->blk[0].n1g, h->blk[0].n1b}, h->X, h->A.hi, h->A.lo, h->A.sf, h->fmt, T, h->J,
                                        h->F * h->J, st));
  return 0;
}
// into block b (1 <= b < nblk): X = Spatial_norm (b - 1 even) / Temporal_norm (b - 1 odd) of X (+ Temporal_pos_embed
// when b == 1) + time vector of block b;  A = norm1 of block b (X)
int postnorm_launch(d3d_handle* h, int b, const float* tv, int64_t tv_stride, int64_t T, cudaStream_t st) {
  const LnParams post = ((b - 1) % 2 == 0) ? LnParams{h->sn_g, h->sn_b} : LnParams{h->tn_g, h->tn_b};
  const Blk& nx = h->blk[b];
  KLP(D3D_PROF_LN, st,
      launch_postnorm_add_ln(h->X, post, (b == 1) ? h->tpos : nullptr, tv ? tv + b * kC : nullptr, tv_stride,
                             LnParams{nx.n1g, nx.n1b}, h->A.hi, h->A.lo, h->A.sf, h->fmt, T, h->J, h->F, st));
  return 0;
}
// A = norm2 of block b (X)
int norm2_launch(d3d_handle* h, int b, int64_t T, cudaStream_t st) {
  KLP(D3D_PROF_LN, st, launch_ln_split(h->X, LnParams{h->blk[b].n2g, h->blk[b].n2b}, 1e-6f, h->A.hi, h->A.lo, h->A.sf, h->fmt,
                                       T, st));
  return 0;
}

// One denoiser evaluation up to (excluding) the final post-norm + head: leaves the residual stream in h->X.
int run_blocks(d3d_handle* h, const float* x2d, const float* y, const float* x5, const float* tv, int64_t tv_stride,
               int B, int n_blocks, cudaStream_t st) {
  const int64_t T = static_cast<int64_t>(B) * h->F * h->J;
  const int gm = h->cfg.gemm_mode, am = h->cfg.attn_mode;
  int r;
  if ((r = lift_launch(h, x2d, y, x5, tv, tv_stride, T, st))) return r;
  for (int b = 0; b < n_blocks; ++b) {
    const Blk& k = h->blk[b];
    const bool spatial = (b % 2) == 0;
    if ((r = run_gemm(h, h->A, k.qkv, T, EPI_QKV16, nullptr, nullptr, nullptr, nullptr, h->QKV, gm, st))) return r;
    if ((r = run_attention(h, h->QKV, h->ATT.hi, h->ATT.lo, nullptr, B, spatial, am, st))) return r;
    if (fuse_ln_enabled() && can_fuse_ln(h, gm)) {        // proj + residual + norm2 (MODEL:127-128) in one kernel
      const LnFuse ln2{k.n2g, k.n2b, 1e-6f, &h->A};
      if ((r = run_gemm(h, h->ATT, k.proj, T, EPI_F32, h->X, h->X, nullptr, nullptr, nullptr, gm, st, &ln2))) return r;
    } else if (h->defer_ln2) {                            // proj + residual emits x as fc1's operand; fc1 applies norm2
      const DeferLn dl{&h->A, h->ln_stats, k.fc1_s, k.fc1_c, 1e-6f};
      if ((r = run_gemm(h, h->ATT, k.proj, T, EPI_F32_EMIT, h->X, h->X, nullptr, nullptr, nullptr, gm, st, nullptr, nullptr, &dl))) return r;
      if ((r = run_gemm(h, h->A, k.fc1, T, EPI_GELU_DLN, nullptr, nullptr, h->H.hi, h->H.lo, nullptr, gm, st, nullptr, h->H.sf, &dl))) return r;
    } else {
      if ((r = run_gemm(h, h->ATT, k.proj, T, EPI_F32, h->X, h->X, nullptr, nullptr, nullptr, gm, st, nullptr, nullptr, nullptr,
                        h->have_m_x ? &h->m_x : nullptr))) return r;
      if ((r = norm2_launch(h, b, T, st))) return r;
    }
    if (!h->defer_ln2 &&
        (r = run_gemm(h, h->A, k.fc1, T, EPI_GELU_SPLIT, nullptr, nullptr, h->H.hi, h->H.lo, nullptr, gm, st, nullptr, h->H.sf))) return r;
    if ((r = run_gemm(h, h->H, k.fc2, T, EPI_F32, h->X, h->X, nullptr, nullptr, nullptr, gm, st, nullptr, nullptr, nullptr,
                      h->have_m_x ? &h->m_x : nullptr))) return r;
    if (b + 1 < n_blocks && (r = postnorm_launch(h, b + 1, tv, tv_stride, T, st))) return r;
  }
  return 0;
}

int run_head(d3d_handle* h, const DdimStep& s, float* y, const float* noise, float* out3, float* trace_y,
             float* trace_x0, int trace_idx, int B, cudaStream_t st) {
  const int64_t T = static_cast<int64_t>(B) * h->F * h->J;
  KLP(D3D_PROF_HEAD, st, launch_head_ddim(h->X, LnParams{h->tn_g, h->tn_b}, LnParams{h->hg, h->hb}, h->wh, h->bh, s,
                                          y, noise, out3, trace_y, trace_x0, h->S, trace_idx, T, st));
  return 0;
}

int ensure_table(d3d_handle* h, cudaStream_t st) {
  if (!h->cfg.with_time_emb) return 0;
  if (h->table_valid) {
    // computed on an earlier caller's stream: order this stream behind it
    CK(cudaStreamWaitEvent(st, h->table_event, 0));
    return 0;
  }
  std::vector<float> tf(h->S);
  for (int i = 0; i < h->S; ++i) tf[i] = static_cast<float>(h->times[i]);
  CK(cudaMemcpyAsync(h->t_f32, tf.data(), sizeof(float) * h->S, cudaMemcpyHostToDevice, st));
  CK(cudaStreamSynchronize(st));   // tf is a stack vector
  int r = compute_time_table(h, h->t_f32, h->S, h->tv_steps, st);
  if (r) return r;
  CK(cudaEventRecord(h->table_event, st));
  h->table_valid = true;
  return 0;
}

// Per-call preparation outside any graph: the spatial tcgen05 attention loads 128-row boxes for 119-token units, so
// the last unit of a batch reads up to 9 rows past T.  They are masked (P = 0), but 0 * Inf/NaN would still poison
// P.V if those rows held non-finite leftovers of an earlier, larger batch: zero them whenever the batch shrank.
int prep_batch(d3d_handle* h, int B, cudaStream_t st) {
  const int64_t T = static_cast<int64_t>(B) * h->F * h->J;
  if (T < h->qkv_rows_dirty) {
    const int64_t rows = std::min<int64_t>(128, h->tok_cap - T);
    if (rows > 0) CK(cudaMemsetAsync(h->QKV + T * kQkvRow, 0, static_cast<size_t>(rows) * kQkvRow * sizeof(__half), st));
  }
  if (T > h->qkv_rows_dirty) h->qkv_rows_dirty = T;
  return 0;
}

// per-sample timesteps (int64, device) -> general time table [B, nblk, 512]; everything stays on the stream
int general_time_table(d3d_handle* h, const int64_t* t_dev, int B, cudaStream_t st) {
  KL(launch_t_to_f32(t_dev, B, h->t_f32, st));
  return compute_time_table(h, h->t_f32, B, h->tv_general, st);
}

int run_sampler(d3d_handle* h, int B, float* trace_y, float* trace_x0, cudaStream_t st) {
  const int64_t n3 = static_cast<int64_t>(B) * h->F * h->J * 3;
  for (int s = 0; s < h->S; ++s) {
    const float* tv = h->cfg.with_time_emb ? h->tv_steps + static_cast<int64_t>(s) * h->nblk * kC : nullptr;
    int r = run_blocks(h, h->in_x2d, h->y, nullptr, tv, 0, B, h->nblk, st);
    if (r) return r;
    const float* nz = (h->need_noise && !h->steps[s].last) ? h->in_noise + static_cast<int64_t>(s) * n3 : nullptr;
    if ((r = run_head(h, h->steps[s], h->y, nz, nullptr, trace_y, trace_x0, s, B, st))) return r;
  }
  return 0;
}

void drop_graphs(d3d_handle* h) {
  for (auto& g : h->graphs) cudaGraphExecDestroy(g.second);
  h->graphs.clear();
  h->graph_launches.clear();
}

int check_ready(d3d_handle* h, int B) {
  if (!h) return -1;
  if (B < 1 || B > h->cfg.max_clips) return fail(h, -2, "B out of range [1, max_clips]");
  return check_weights(h);
}

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    int cur = -1;
    cudaGetDevice(&cur);
    if (prev >= 0 && cur != prev) cudaSetDevice(prev);
  }
};

}  // namespace

// =====================================================================================================
extern "C" {

int d3d_abi_version(void) { return D3D_ABI_VERSION; }

const char* d3d_last_error(const d3d_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int64_t d3d_launch_count(const d3d_handle* h) { return h ? h->launches : 0; }

int64_t d3d_workspace_bytes(const d3d_handle* h) { return h ? h->alloc_bytes : 0; }

int d3d_create(const d3d_config* cfg, d3d_handle** out) {
  if (!cfg || !out) { g_create_error = "null argument"; return -1; }
  *out = nullptr;
  if (cfg->embed_dim != kC || cfg->num_heads != kHeads || cfg->mlp_hidden != kHidden) {
    g_create_error = "unsupported shape: kernels are specialised for embed_dim 512, 8 heads, mlp hidden 1024";
    return -3;
  }
  if (cfg->num_frame < 1 || cfg->num_frame > 256 || cfg->num_joints < 1 || cfg->num_joints > 32 || cfg->depth < 1 ||
      cfg->depth > 64 || cfg->max_clips < 1) {
    g_create_error = "unsupported shape: need 1<=F<=256, 1<=J<=32, 1<=depth<=64, max_clips>=1";
    return -3;
  }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e) + " (this library has no CPU fallback)";
    return e != cudaSuccess ? static_cast<int>(e) : -4;
  }
  if (cfg->device < 0 || cfg->device >= ndev) { g_create_error = "bad device ordinal"; return -2; }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, cfg->device);
  if (prop.major != 10) {
    g_create_error = "device is not sm_100 (Blackwell B200); this library is sm_100a-only";
    return -5;
  }
  DeviceGuard guard(cfg->device);
  d3d_handle* h = new d3d_handle();
  h->cfg = *cfg;
  h->fmt = mode_fmt(cfg->gemm_mode);
  // OFF by default (D3D_DEFER_LN2=1 enables it): measured on B200 at cfg3 (profiles/r02j_*): with the residual update of
  // proj done by the L2 (EPI_F32_RED) the separate norm2 pass is cheaper than the emitting epilogue, which has to pull
  // the residual rows into the SM -- 3183 ms per step (RED + norm2 kernel) against 3217 ms (EMIT + DLN)
  h->defer_ln2 = cfg->gemm_mode == D3D_GEMM_TC_F4C && env_int("D3D_DEFER_LN2", 0) == 1 && pick_cg(kC) == 2;
  h->F = cfg->num_frame;
  h->J = cfg->num_joints;
  h->nblk = 2 * cfg->depth;
  h->num_sms = prop.multiProcessorCount;
  h->blk.resize(h->nblk);
  const int64_t T = static_cast<int64_t>(cfg->max_clips) * h->F * h->J;
  h->tok_cap = (T + 511) / 512 * 512;

  auto body = [&]() -> int {
    int r;
    CK(cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&h->table_event, cudaEventDisableTiming));
    if ((r = dev_alloc(h, &h->absmax_dev, 2))) return r;
    if ((r = dev_alloc(h, &h->vel_tmp, 2))) return r;
    CK(configure_gemm_tc());
    CK(configure_attention());
    CK(configure_attention_mma());
    CK(configure_attention_tc());
    for (auto& b : h->blk) {
      if ((r = alloc_lin(h, &b.qkv, 3 * kC, kC))) return r;
      if ((r = alloc_lin(h, &b.proj, kC, kC))) return r;
      if ((r = alloc_lin(h, &b.fc1, kHidden, kC))) return r;
      if ((r = alloc_lin(h, &b.fc2, kC, kHidden))) return r;
      for (float** p : {&b.n1g, &b.n1b, &b.n2g, &b.n2b, &b.tb})
        if ((r = dev_alloc(h, p, kC))) return r;
      if ((r = dev_alloc(h, &b.tw, static_cast<int64_t>(kC) * 2 * kC))) return r;
      if (h->defer_ln2) {
        if ((r = dev_alloc(h, &b.fc1_raw, static_cast<int64_t>(kHidden) * kC))) return r;
        if ((r = dev_alloc(h, &b.fc1_s, kHidden))) return r;
        if ((r = dev_alloc(h, &b.fc1_c, kHidden))) return r;
      }
    }
    for (float** p : {&h->bf, &h->sn_g, &h->sn_b, &h->tn_g, &h->tn_b, &h->hg, &h->hb})
      if ((r = dev_alloc(h, p, kC))) return r;
    if ((r = dev_alloc(h, &h->wf_t, 5 * kC))) return r;
    if ((r = dev_alloc(h, &h->spos, static_cast<int64_t>(h->J) * kC))) return r;
    if ((r = dev_alloc(h, &h->tpos, static_cast<int64_t>(h->F) * kC))) return r;
    if ((r = dev_alloc(h, &h->wh, 3 * kC))) return r;
    if ((r = dev_alloc(h, &h->bh, 4))) return r;
    if ((r = dev_alloc(h, &h->tm1w, static_cast<int64_t>(2 * kC) * kC))) return r;
    if ((r = dev_alloc(h, &h->tm1b, 2 * kC))) return r;
    if ((r = dev_alloc(h, &h->tm3w, static_cast<int64_t>(2 * kC) * 2 * kC))) return r;
    if ((r = dev_alloc(h, &h->tm3b, 2 * kC))) return r;
    if ((r = dev_alloc(h, &h->perm_dev, 64))) return r;

    if ((r = dev_alloc(h, &h->X, h->tok_cap * kC))) return r;
    if (make_f32_tile_map(&h->m_x, h->X, h->tok_cap, kC)) return fail(h, -20, "cuTensorMapEncodeTiled failed for X");
    h->have_m_x = true;
    if ((r = dev_alloc(h, &h->QKV, h->tok_cap * kQkvRow))) return r;
    if ((r = alloc_operand(h, &h->A, h->tok_cap, kC))) return r;
    if ((r = alloc_operand(h, &h->ATT, h->tok_cap, kC))) return r;
    if ((r = alloc_operand(h, &h->H, h->tok_cap, kHidden))) return r;
    if (h->defer_ln2 && (r = dev_alloc(h, &h->ln_stats, 8 * h->tok_cap))) return r;
    if (h->J == 17) {
      if (make_attn_tc_maps_spatial(&h->attn_sp, h->QKV, h->ATT.hi, h->ATT.lo, h->fmt, h->tok_cap, h->F))
        return fail(h, -20, "cuTensorMapEncodeTiled failed for the spatial-attention maps");
      h->have_attn_sp = true;
    }
    {   // every F <= 256 runs on the tcgen05 kernel (F <= 64: 2 or 4 joints packed per 128-row tile)
      if (make_attn_tc_maps(&h->attn_tc, h->QKV, h->ATT.hi, h->ATT.lo, h->fmt, h->F, h->J, cfg->max_clips))
        return fail(h, -20, "cuTensorMapEncodeTiled failed for the temporal-attention maps");
      h->have_attn_tc = true;
    }
    if ((r = dev_alloc(h, &h->in_x2d, T * 2))) return r;
    if ((r = dev_alloc(h, &h->y, T * 3))) return r;
    h->t_rows_cap = cfg->max_clips > 1024 ? cfg->max_clips : 1024;
    if ((r = dev_alloc(h, &h->t_f32, h->t_rows_cap))) return r;
    if ((r = dev_alloc(h, &h->e0, static_cast<int64_t>(h->t_rows_cap) * kC))) return r;
    if ((r = dev_alloc(h, &h->h1, static_cast<int64_t>(h->t_rows_cap) * 2 * kC))) return r;
    if ((r = dev_alloc(h, &h->h2, static_cast<int64_t>(h->t_rows_cap) * 2 * kC))) return r;
    if ((r = dev_alloc(h, &h->tv_general, static_cast<int64_t>(cfg->max_clips) * h->nblk * kC))) return r;
    CK(cudaDeviceSynchronize());
    return 0;
  };
  int r = body();
  if (r) {
    g_create_error = h->err;
    d3d_destroy(h);
    return r;
  }
  *out = h;
  return 0;
}

void d3d_destroy(d3d_handle* h) {
  if (!h) return;
  DeviceGuard guard(h->cfg.device);
  cudaDeviceSynchronize();
  drop_graphs(h);
  for (void* p : h->allocs) cudaFree(p);
  for (cudaEvent_t e : h->prof_pool) cudaEventDestroy(e);
  if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
  if (h->table_event) cudaEventDestroy(h->table_event);
  delete h;
}

int d3d_load_weights(d3d_handle* h, const d3d_tensor* tensors, int32_t n) {
  if (!h || !tensors) return -1;
  DeviceGuard guard(h->cfg.device);
  CK(cudaDeviceSynchronize());   // in-flight work on any (non-blocking) stream may still read the packed weights
  drop_graphs(h);
  h->table_valid = false;
  float* stage = nullptr;   // device staging for tensors that need a transform
  const int64_t stage_cap = static_cast<int64_t>(3 * kC) * kHidden;
  CK(cudaMalloc(&stage, stage_cap * sizeof(float)));
  struct Free { float* p; ~Free() { cudaFree(p); } } free_stage{stage};

  auto copy_to = [&](float* dst, const d3d_tensor& t, int64_t expect) -> int {
    if (t.numel != expect)
      return fail(h, -10, std::string("tensor '") + t.name + "' has " + std::to_string(t.numel) + " elements, expected " +
                              std::to_string(expect));
    CK(cudaMemcpy(dst, t.data, expect * sizeof(float), t.on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
    return 0;
  };
  // split the fp32 weight in `stage` into the operand arrays of l, with the range guard
  auto split_stage = [&](Lin& l, const std::string& tname) -> int {
    CK(cudaMemset(h->absmax_dev, 0, 2 * sizeof(float)));
    CK(launch_split(stage, l.hi, l.lo, l.sf, l.N, l.K, h->fmt, 1, 0, h->absmax_dev));
    CK(cudaDeviceSynchronize());
    // range guard (SURVEY.md 7.3-1): the main operand is fp16 and the correction operands are scaled images of it, so a
    // weight beyond the fp16 range (or a non-finite one) would silently become Inf inside every GEMM.  [0] = max |w|
    // over finite values, [1] = 1 when a NaN / Inf was seen.
    float am[2] = {0.f, 0.f};
    CK(cudaMemcpy(am, h->absmax_dev, sizeof(am), cudaMemcpyDeviceToHost));
    if (am[1] != 0.f) return fail(h, -12, std::string("tensor '") + tname + "' holds NaN / Inf");
    if (am[0] > kMaxWeightAbs)
      return fail(h, -12, std::string("tensor '") + tname + "': max |w| = " + std::to_string(am[0]) +
                              " exceeds the fp16 operand range (" + std::to_string(kMaxWeightAbs) + ")");
    l.have_w = true;
    return 0;
  };
  auto load_lin_w = [&](Lin& l, const d3d_tensor& t) -> int {
    int r = copy_to(stage, t, static_cast<int64_t>(l.N) * l.K);
    if (r) return r;
    return split_stage(l, t.name);
  };

  for (int i = 0; i < n; ++i) {
    const d3d_tensor& t = tensors[i];
    if (!t.name || !t.data) return fail(h, -1, "null tensor name/data");
    std::string name = t.name;
    if (name.rfind("module.", 0) == 0) name = name.substr(7);
    if (name.rfind("model.", 0) == 0) name = name.substr(6);
    int r = 0;
    if (name == "fusion_layer.weight") {           // [512,5] -> transposed [5][512]
      std::vector<float> w(5 * kC), wt(5 * kC);
      if (t.numel != 5 * kC) return fail(h, -10, "fusion_layer.weight must be [512,5]");
      CK(cudaMemcpy(w.data(), t.data, sizeof(float) * 5 * kC, t.on_device ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost));
      for (int c = 0; c < kC; ++c)
        for (int k = 0; k < 5; ++k) wt[k * kC + c] = w[c * 5 + k];
      CK(cudaMemcpy(h->wf_t, wt.data(), sizeof(float) * 5 * kC, cudaMemcpyHostToDevice));
    } else if (name == "fusion_layer.bias") r = copy_to(h->bf, t, kC);
    else if (name == "Spatial_pos_embed") r = copy_to(h->spos, t, static_cast<int64_t>(h->J) * kC);
    else if (name == "Temporal_pos_embed") r = copy_to(h->tpos, t, static_cast<int64_t>(h->F) * kC);
    else if (name == "Spatial_norm.weight") r = copy_to(h->sn_g, t, kC);
    else if (name == "Spatial_norm.bias") r = copy_to(h->sn_b, t, kC);
    else if (name == "Temporal_norm.weight") r = copy_to(h->tn_g, t, kC);
    else if (name == "Temporal_norm.bias") r = copy_to(h->tn_b, t, kC);
    else if (name == "head.0.weight") r = copy_to(h->hg, t, kC);
    else if (name == "head.0.bias") r = copy_to(h->hb, t, kC);
    else if (name == "head.1.weight") r = copy_to(h->wh, t, 3 * kC);
    else if (name == "head.1.bias") r = copy_to(h->bh, t, 3);
    else if (name == "time_mlp.1.weight") r = copy_to(h->tm1w, t, static_cast<int64_t>(2 * kC) * kC);
    else if (name == "time_mlp.1.bias") r = copy_to(h->tm1b, t, 2 * kC);
    else if (name == "time_mlp.3.weight") r = copy_to(h->tm3w, t, static_cast<int64_t>(2 * kC) * 2 * kC);
    else if (name == "time_mlp.3.bias") r = copy_to(h->tm3b, t, 2 * kC);
    else if (name.rfind("STEblocks.", 0) == 0 || name.rfind("TTEblocks.", 0) == 0) {
      const bool spatial = name[0] == 'S';
      const size_t dot = name.find('.', 10);
      if (dot == std::string::npos) return fail(h, -11, "unknown tensor '" + name + "'");
      const int idx = atoi(name.substr(10, dot - 10).c_str());
      if (idx < 0 || idx >= h->cfg.depth) return fail(h, -11, "block index out of range in '" + name + "'");
      Blk& b = h->blk[2 * idx + (spatial ? 0 : 1)];
      const std::string sub = name.substr(dot + 1);
      if (sub == "norm1.weight") r = copy_to(b.n1g, t, kC);
      else if (sub == "norm1.bias") r = copy_to(b.n1b, t, kC);
      else if (sub == "norm2.weight") { r = copy_to(b.n2g, t, kC); b.fold_dirty = h->defer_ln2; }
      else if (sub == "norm2.bias") { r = copy_to(b.n2b, t, kC); b.fold_dirty = h->defer_ln2; }
      else if (sub == "attn.qkv.weight") r = load_lin_w(b.qkv, t);
      else if (sub == "attn.qkv.bias") r = copy_to(b.qkv.bias, t, 3 * kC);
      else if (sub == "attn.proj.weight") r = load_lin_w(b.proj, t);
      else if (sub == "attn.proj.bias") r = copy_to(b.proj.bias, t, kC);
      else if (sub == "mlp.fc1.weight") {
        if (h->defer_ln2) { r = copy_to(b.fc1_raw, t, static_cast<int64_t>(kHidden) * kC); b.fold_dirty = true; }
        else r = load_lin_w(b.fc1, t);
      } else if (sub == "mlp.fc1.bias") { r = copy_to(b.fc1.bias, t, kHidden); b.fold_dirty = h->defer_ln2; }
      else if (sub == "mlp.fc2.weight") r = load_lin_w(b.fc2, t);
      else if (sub == "mlp.fc2.bias") r = copy_to(b.fc2.bias, t, kC);
      else if (sub == "time_mlp.1.weight") r = copy_to(b.tw, t, static_cast<int64_t>(kC) * 2 * kC);
      else if (sub == "time_mlp.1.bias") r = copy_to(b.tb, t, kC);
      else return fail(h, -11, "unknown tensor '" + name + "'");
    } else {
      return fail(h, -11, "unknown tensor '" + name + "'");
    }
    if (r) return r;
    h->loaded[name] = true;
  }
  // deferred norm2: (re)fold every block whose norm2 / fc1 tensors changed, once all four are present
  for (int bi = 0; bi < h->nblk; ++bi) {
    Blk& b = h->blk[bi];
    if (!b.fold_dirty) continue;
    const std::string pre = std::string(bi % 2 == 0 ? "STEblocks." : "TTEblocks.") + std::to_string(bi / 2) + ".";
    bool all = true;
    for (const char* s : {"norm2.weight", "norm2.bias", "mlp.fc1.weight", "mlp.fc1.bias"}) all = all && h->loaded.count(pre + s);
    if (!all) continue;
    CK(launch_fold_ln_linear(b.fc1_raw, b.n2g, b.n2b, b.fc1.bias, stage, b.fc1_s, b.fc1_c, kHidden, kC, 0));
    int r = split_stage(b.fc1, pre + "mlp.fc1.weight (folded with norm2.weight)");
    if (r) return r;
    b.fold_dirty = false;
  }
  CK(cudaDeviceSynchronize());
  return 0;
}

int d3d_set_schedule(d3d_handle* h, int32_t S, const int32_t* times, const float* ac, const float* s1m, int32_t T,
                     float eta, int32_t clip_denoised) {
  if (!h || !times || !ac || !s1m) return -1;
  if (S < 1 || S > 1024) return fail(h, -2, "sampling_timesteps out of range [1,1024]");
  DeviceGuard guard(h->cfg.device);
  // a failed call must not leave a half-written schedule behind: nothing is usable until everything validated
  h->have_schedule = false;
  drop_graphs(h);
  h->table_valid = false;
  if (S > h->t_rows_cap) return fail(h, -2, "sampling_timesteps exceeds the time-MLP scratch rows");
  std::vector<DdimStep> steps(S);
  bool need_noise = false;
  for (int i = 0; i < S; ++i) {
    const int t = times[i], tn = times[i + 1];
    if (t < 0 || t >= T || tn >= T) return fail(h, -2, "time index outside the schedule buffers");
    DdimStep s{};
    s.clip = clip_denoised ? 1 : 0;
    if (tn < 0) {
      s.last = 1;                                   // DIFF:283-285
    } else {
      // DIFF:287-292 evaluated in fp32, one rounding per op as torch does on 0-dim fp32 tensors
      const volatile float alpha = ac[t], alpha_next = ac[tn];
      volatile float q = alpha / alpha_next;
      volatile float a1 = 1.0f - q;
      volatile float a2 = 1.0f - alpha_next;
      volatile float a3 = a1 * a2;
      volatile float a4 = 1.0f - alpha;
      volatile float a5 = a3 / a4;
      volatile float sig = eta * sqrtf(a5);
      volatile float s2 = sig * sig;
      volatile float c0 = a2 - s2;
      s.sigma = sig;
      s.c = sqrtf(c0);
      s.alpha = alpha;
      s.sqrt_alpha_next = sqrtf(alpha_next);
      s.sqrt_one_minus = s1m[t];
      if (s.sigma != 0.0f) need_noise = true;
    }
    steps[i] = s;
  }
  if (S > h->tv_cap) {
    CK(cudaDeviceSynchronize());     // the old table may still be read by in-flight work
    int r = dev_alloc(h, &h->tv_steps, static_cast<int64_t>(S) * h->nblk * kC);
    if (r) return r;
    h->tv_cap = S;
  }
  h->S = S;
  h->times.assign(times, times + S + 1);
  h->steps.swap(steps);
  h->need_noise = need_noise;
  h->have_schedule = true;
  return 0;
}

int d3d_forward_denoise(d3d_handle* h, const float* x5, const int64_t* t_dev, float* out3, int32_t B, void* stream) {
  int r = check_ready(h, B);
  if (r) return r;
  if (!x5 || !out3 || (h->cfg.with_time_emb && !t_dev)) return fail(h, -1, "null argument");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float* tv = nullptr;
  if ((r = prep_batch(h, B, st))) return r;
  if (h->cfg.with_time_emb) {
    // per-sample t (the p_losses call of DIFF:392-419): converted and embedded on the device, no host round trip
    if ((r = general_time_table(h, t_dev, B, st))) return r;
    tv = h->tv_general;
  }
  if ((r = run_blocks(h, nullptr, nullptr, x5, tv, static_cast<int64_t>(h->nblk) * kC, B, h->nblk, st))) return r;
  DdimStep s{};
  return run_head(h, s, nullptr, nullptr, out3, nullptr, nullptr, 0, B, st);
}

int d3d_debug_forward_blocks(d3d_handle* h, const float* x5, const int64_t* t_dev, int32_t B, int32_t n_blocks,
                             float* x_out, void* stream) {
  int r = check_ready(h, B);
  if (r) return r;
  if (n_blocks < 0 || n_blocks > h->nblk) return fail(h, -2, "n_blocks out of range");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float* tv = nullptr;
  if ((r = prep_batch(h, B, st))) return r;
  if (h->cfg.with_time_emb) {
    if (!t_dev) return fail(h, -1, "null argument");
    if ((r = general_time_table(h, t_dev, B, st))) return r;
    tv = h->tv_general;
  }
  if ((r = run_blocks(h, nullptr, nullptr, x5, tv, static_cast<int64_t>(h->nblk) * kC, B, n_blocks, st))) return r;
  const int64_t T = static_cast<int64_t>(B) * h->F * h->J;
  CK(cudaMemcpyAsync(x_out, h->X, sizeof(float) * T * kC, cudaMemcpyDeviceToDevice, st));
  return 0;
}

static int sample_on_device(d3d_handle* h, int B, float* trace_y, float* trace_x0, cudaStream_t st) {
  int r = ensure_table(h, st);
  if (r) return r;
  const bool tracing = trace_y || trace_x0;
  if (!h->cfg.use_graph || tracing || h->prof) return run_sampler(h, B, trace_y, trace_x0, st);
  auto it = h->graphs.find(B);
  if (it == h->graphs.end()) {
    const int64_t before = h->launches;
    cudaGraph_t graph = nullptr;
    CK(cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeThreadLocal));
    r = run_sampler(h, B, nullptr, nullptr, h->cap_stream);
    cudaError_t e = cudaStreamEndCapture(h->cap_stream, &graph);
    const int64_t n_kernels = h->launches - before;
    h->launches = before;
    if (r) { if (graph) cudaGraphDestroy(graph); return r; }
    CK(e);
    cudaGraphExec_t exec = nullptr;
    e = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    CK(e);
    h->graphs[B] = exec;
    h->graph_launches[B] = n_kernels;
    it = h->graphs.find(B);
  }
  CK(cudaGraphLaunch(it->second, st));
  h->launches += h->graph_launches[B];
  return 0;
}

static int ensure_noise_buf(d3d_handle* h, int B) {
  const int64_t need = static_cast<int64_t>(h->S - 1) * B * h->F * h->J * 3;
  if (need > h->in_noise_cap) {
    drop_graphs(h);
    int r = dev_alloc(h, &h->in_noise, need, false);
    if (r) return r;
    h->in_noise_cap = need;
  }
  return 0;
}

int d3d_ddim_sample(d3d_handle* h, const float* x2d, const float* noise0, const float* step_noise, float* y0,
                    float* trace_y, float* trace_x0, int32_t B, void* stream) {
  int r = check_ready(h, B);
  if (r) return r;
  if (!h->have_schedule) return fail(h, -31, "d3d_set_schedule has not been called");
  if (!x2d || !noise0 || !y0) return fail(h, -1, "null argument");
  if (h->need_noise && !step_noise && h->S > 1) return fail(h, -1, "eta != 0 requires step_noise");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t T = static_cast<int64_t>(B) * h->F * h->J;
  if ((r = prep_batch(h, B, st))) return r;
  CK(cudaMemcpyAsync(h->in_x2d, x2d, sizeof(float) * T * 2, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(h->y, noise0, sizeof(float) * T * 3, cudaMemcpyDeviceToDevice, st));
  if (h->need_noise && h->S > 1) {
    if ((r = ensure_noise_buf(h, B))) return r;
    CK(cudaMemcpyAsync(h->in_noise, step_noise, sizeof(float) * T * 3 * (h->S - 1), cudaMemcpyDeviceToDevice, st));
  }
  if ((r = sample_on_device(h, B, trace_y, trace_x0, st))) return r;
  CK(cudaMemcpyAsync(y0, h->y, sizeof(float) * T * 3, cudaMemcpyDeviceToDevice, st));
  return 0;
}

int d3d_ddim_sample_host(d3d_handle* h, const float* x2d, const float* noise0, const float* step_noise, float* y0,
                         int32_t B, void* stream) {
  int r = check_ready(h, B);
  if (r) return r;
  if (!h->have_schedule) return fail(h, -31, "d3d_set_schedule has not been called");
  if (!x2d || !noise0 || !y0) return fail(h, -1, "null argument");
  if (h->need_noise && !step_noise && h->S > 1) return fail(h, -1, "eta != 0 requires step_noise");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t T = static_cast<int64_t>(B) * h->F * h->J;
  if ((r = prep_batch(h, B, st))) return r;
  CK(cudaMemcpyAsync(h->in_x2d, x2d, sizeof(float) * T * 2, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(h->y, noise0, sizeof(float) * T * 3, cudaMemcpyHostToDevice, st));
  if (h->need_noise && h->S > 1) {
    if ((r = ensure_noise_buf(h, B))) return r;
    CK(cudaMemcpyAsync(h->in_noise, step_noise, sizeof(float) * T * 3 * (h->S - 1), cudaMemcpyHostToDevice, st));
  }
  if ((r = sample_on_device(h, B, nullptr, nullptr, st))) return r;
  CK(cudaMemcpyAsync(y0, h->y, sizeof(float) * T * 3, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}

static int upload_perm(d3d_handle* h, const int32_t* left, const int32_t* right, int32_t n_lr, cudaStream_t st);

int d3d_window_gather(d3d_handle* h, const float* seq2d, const int64_t* win_start, int64_t n_win, const int32_t* left,
                      const int32_t* right, int32_t n_lr, float* x2d_out, float* x2d_flip_out, void* stream) {
  if (!h || !seq2d || !win_start || !x2d_out) return -1;
  if (n_win < 0) return fail(h, -2, "n_win < 0");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (x2d_flip_out) {
    int r = upload_perm(h, left, right, n_lr, st);
    if (r) return r;
  }
  KL(launch_window_gather(seq2d, win_start, h->perm_dev, x2d_out, x2d_flip_out, n_win, h->F, h->J, st));
  return 0;
}

int d3d_window_scatter(d3d_handle* h, const float* pred, const int64_t* win_start, const int32_t* first_valid,
                       int64_t n_win, float* seq3d_out, void* stream) {
  if (!h || !pred || !win_start || !first_valid || !seq3d_out) return -1;
  if (n_win < 0) return fail(h, -2, "n_win < 0");
  DeviceGuard guard(h->cfg.device);
  KL(launch_window_scatter(pred, win_start, first_valid, seq3d_out, n_win, h->F, h->J, static_cast<cudaStream_t>(stream)));
  return 0;
}

// joint permutation of a horizontal flip (new[left[i]] = old[right[i]] and vice versa, RUN:584-585): uploaded only
// when the lists change
static int upload_perm(d3d_handle* h, const int32_t* left, const int32_t* right, int32_t n_lr, cudaStream_t st) {
  if (n_lr < 0 || n_lr > 16 || (n_lr > 0 && (!left || !right))) return fail(h, -2, "bad joint lists");
  int32_t perm[64];
  for (int j = 0; j < 64; ++j) perm[j] = j;
  for (int i = 0; i < n_lr; ++i) {
    if (left[i] < 0 || left[i] >= h->J || right[i] < 0 || right[i] >= h->J) return fail(h, -2, "joint index out of range");
    perm[left[i]] = right[i];
    perm[right[i]] = left[i];
  }
  if (!h->perm_valid || memcmp(perm, h->perm_host, sizeof(perm)) != 0) {
    CK(cudaStreamSynchronize(st));
    CK(cudaMemcpy(h->perm_dev, perm, sizeof(perm), cudaMemcpyHostToDevice));
    memcpy(h->perm_host, perm, sizeof(perm));
    h->perm_valid = true;
  }
  return 0;
}

int d3d_tta_merge(d3d_handle* h, const float* y, const float* yf, const int32_t* left, const int32_t* right,
                  int32_t n_lr, float scale, float* out, int64_t n_frames, void* stream) {
  if (!h || !y || !yf || !out) return -1;
  if (n_lr < 0 || n_lr > 16 || (n_lr > 0 && (!left || !right))) return fail(h, -2, "bad joint lists");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int32_t perm[64];
  for (int j = 0; j < 64; ++j) perm[j] = j;
  for (int i = 0; i < n_lr; ++i) {
    if (left[i] < 0 || left[i] >= h->J || right[i] < 0 || right[i] >= h->J) return fail(h, -2, "joint index out of range");
    perm[left[i]] = right[i];      // new[left] = old[right]  (RUN:584-585)
    perm[right[i]] = left[i];
  }
  if (!h->perm_valid || memcmp(perm, h->perm_host, sizeof(perm)) != 0) {      // upload only when the lists change
    CK(cudaStreamSynchronize(st));
    CK(cudaMemcpy(h->perm_dev, perm, sizeof(perm), cudaMemcpyHostToDevice));
    memcpy(h->perm_host, perm, sizeof(perm));
    h->perm_valid = true;
  }
  KL(launch_tta_merge(y, yf, h->perm_dev, scale, out, n_frames, h->J, st));
  return 0;
}

int d3d_mpjpe_accumulate(d3d_handle* h, const float* pred, const float* gt, const uint8_t* mask, int64_t n_frames,
                         double* acc, void* stream) {
  if (!h || !pred || !gt || !acc) return -1;
  DeviceGuard guard(h->cfg.device);
  KL(launch_mpjpe(pred, gt, mask, n_frames, h->J, acc, static_cast<cudaStream_t>(stream)));
  return 0;
}

int d3d_pose_metrics_accumulate(d3d_handle* h, const float* pred, const float* gt, const int64_t* frame_index,
                                int64_t n_sel, double* acc, void* stream) {
  if (!h || !pred || !gt || !acc) return -1;
  if (n_sel < 0) return fail(h, -2, "n_sel < 0");
  DeviceGuard guard(h->cfg.device);
  KL(launch_pose_metrics(pred, gt, frame_index, n_sel, h->J, acc, h->vel_tmp, static_cast<cudaStream_t>(stream)));
  return 0;
}

int d3d_profile_begin(d3d_handle* h) {
  if (!h) return -1;
  h->prof = true;
  h->prof_recs.clear();
  h->prof_next = 0;
  return 0;
}

int d3d_profile_end(d3d_handle* h, double* ms_per_class, int64_t* launches_per_class) {
  if (!h || !ms_per_class || !launches_per_class) return -1;
  DeviceGuard guard(h->cfg.device);
  h->prof = false;
  CK(cudaDeviceSynchronize());
  for (int c = 0; c < D3D_PROF_NUM_CLASSES; ++c) { ms_per_class[c] = 0.0; launches_per_class[c] = 0; }
  for (auto& r : h->prof_recs) {
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, r.a, r.b));
    ms_per_class[r.cls] += ms;
    launches_per_class[r.cls] += 1;
  }
  h->prof_recs.clear();
  h->prof_next = 0;
  return 0;
}

// ------------------------------------------------------------------------------------ kernel-level entry points
int d3d_op_layernorm(d3d_handle* h, const float* x, const float* gamma, const float* beta, float eps, float* out,
                     int64_t rows, void* stream) {
  if (!h || !x || !gamma || !beta || !out) return -1;
  DeviceGuard guard(h->cfg.device);
  KL(launch_ln_f32(x, LnParams{gamma, beta}, eps, out, rows, static_cast<cudaStream_t>(stream)));
  return 0;
}

int d3d_op_attention(d3d_handle* h, const float* qkv, float* out, int32_t B, int32_t spatial, int32_t attn_mode,
                     void* stream) {
  if (!h || !qkv || !out) return -1;
  if (B < 1 || B > h->cfg.max_clips) return fail(h, -2, "B out of range [1, max_clips]");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // the hot path receives q | k | v_hi | v_lo fp16 rows from the qkv GEMM epilogue; here they are packed from fp32
  { int r0 = prep_batch(h, B, st); if (r0) return r0; }
  KL(launch_pack_qkv16(qkv, h->QKV, static_cast<int64_t>(B) * h->F * h->J, st));
  return run_attention(h, h->QKV, nullptr, nullptr, out, B, spatial != 0, attn_mode, st);
}

// rows [0, T) of a [tok_cap, 512] workspace operand -> raw arrays (layout: include/diff3d_b200.h,
// d3d_debug_attention_operand)
static int copy_operand_out(d3d_handle* h, const OperandBuf& o, int64_t T, void* hi_out, void* second_out, cudaStream_t st) {
  CK(cudaMemcpyAsync(hi_out, o.hi, static_cast<size_t>(T) * kC * 2, cudaMemcpyDeviceToDevice, st));
  if (h->fmt == FMT_F4C) {
    // second_out: [T][512] c4 bytes (256 B of P nibbles | 256 B of Q nibbles), then [T][32] scale bytes, row-major
    CK(cudaMemcpyAsync(second_out, o.lo, static_cast<size_t>(T) * kC, cudaMemcpyDeviceToDevice, st));
    KL(launch_sf_rows(o.sf, static_cast<uint8_t*>(second_out) + static_cast<size_t>(T) * kC, T, kC, st));
  } else {
    CK(cudaMemcpyAsync(second_out, o.lo, static_cast<size_t>(T) * kC * 2, cudaMemcpyDeviceToDevice, st));
  }
  return 0;
}

int d3d_debug_attention_operand(d3d_handle* h, const float* qkv, void* hi_out, void* second_out, int32_t B,
                                int32_t spatial, int32_t attn_mode, void* stream) {
  if (!h || !qkv || !hi_out || !second_out) return -1;
  if (B < 1 || B > h->cfg.max_clips) return fail(h, -2, "B out of range [1, max_clips]");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t T = static_cast<int64_t>(B) * h->F * h->J;
  { int r0 = prep_batch(h, B, st); if (r0) return r0; }
  KL(launch_pack_qkv16(qkv, h->QKV, T, st));
  int r = run_attention(h, h->QKV, h->ATT.hi, h->ATT.lo, nullptr, B, spatial != 0, attn_mode, st);
  if (r) return r;
  return copy_operand_out(h, h->ATT, T, hi_out, second_out, st);
}

int d3d_debug_rowwise(d3d_handle* h, int32_t op, int32_t block, const float* in, const int64_t* t_dev, int32_t shared_t,
                      int32_t B, float* out, void* hi_out, void* second_out, void* stream) {
  int r = check_ready(h, B);
  if (r) return r;
  if (op < D3D_ROWWISE_LIFT || op > D3D_ROWWISE_HEAD) return fail(h, -2, "op out of range");
  const bool operand = op != D3D_ROWWISE_HEAD, timed = op == D3D_ROWWISE_LIFT || op == D3D_ROWWISE_POSTNORM;
  if (!in || (op != D3D_ROWWISE_NORM2 && !out) || (operand && (!hi_out || !second_out)) ||
      (timed && h->cfg.with_time_emb && !t_dev))
    return fail(h, -1, "null argument");
  if (op == D3D_ROWWISE_POSTNORM && (block < 1 || block >= h->nblk)) return fail(h, -2, "block out of range [1, 2 depth)");
  if (op == D3D_ROWWISE_NORM2 && (block < 0 || block >= h->nblk)) return fail(h, -2, "block out of range [0, 2 depth)");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t T = static_cast<int64_t>(B) * h->F * h->J;
  const size_t x_bytes = static_cast<size_t>(T) * kC * sizeof(float);
  const float* tv = nullptr;
  int64_t tv_stride = 0;
  if (timed && h->cfg.with_time_emb) {
    if ((r = general_time_table(h, t_dev, B, st))) return r;
    tv = h->tv_general;
    tv_stride = shared_t ? 0 : static_cast<int64_t>(h->nblk) * kC;
  }
  if (operand) {
    // rows the launch does not write come back as NaN halves / 0xff bytes; the scale atoms (which interleave the
    // padding rows of the last tile) get byte 1, a scale of 2^-126 that no LayerNorm block produces
    CK(cudaMemsetAsync(h->A.hi, 0xff, static_cast<size_t>(T) * kC * 2, st));
    CK(cudaMemsetAsync(h->A.lo, 0xff, static_cast<size_t>(T) * (h->fmt == FMT_F4C ? kC : 2 * kC), st));
    if (h->fmt == FMT_F4C)
      CK(cudaMemsetAsync(h->A.sf, 1, static_cast<size_t>((T + 127) / 128) * 128 * (kC / 16), st));
  }
  if (op == D3D_ROWWISE_LIFT) {
    CK(cudaMemsetAsync(h->X, 0xff, x_bytes, st));
    if (shared_t) {        // the sampler's form: 2D keypoints and the noisy pose in two arrays
      CK(cudaMemcpy2DAsync(h->in_x2d, 2 * sizeof(float), in, 5 * sizeof(float), 2 * sizeof(float), static_cast<size_t>(T),
                           cudaMemcpyDeviceToDevice, st));
      CK(cudaMemcpy2DAsync(h->y, 3 * sizeof(float), in + 2, 5 * sizeof(float), 3 * sizeof(float), static_cast<size_t>(T),
                           cudaMemcpyDeviceToDevice, st));
      r = lift_launch(h, h->in_x2d, h->y, nullptr, tv, tv_stride, T, st);
    } else {               // forward_denoise's form: x5 [T, 5]
      r = lift_launch(h, nullptr, nullptr, in, tv, tv_stride, T, st);
    }
  } else {
    CK(cudaMemcpyAsync(h->X, in, x_bytes, cudaMemcpyDeviceToDevice, st));
    if (op == D3D_ROWWISE_POSTNORM) r = postnorm_launch(h, block, tv, tv_stride, T, st);
    else if (op == D3D_ROWWISE_NORM2) r = norm2_launch(h, block, T, st);
    else r = run_head(h, DdimStep{}, nullptr, nullptr, out, nullptr, nullptr, 0, B, st);
  }
  if (r) return r;
  if (op == D3D_ROWWISE_LIFT || op == D3D_ROWWISE_POSTNORM) CK(cudaMemcpyAsync(out, h->X, x_bytes, cudaMemcpyDeviceToDevice, st));
  return operand ? copy_operand_out(h, h->A, T, hi_out, second_out, st) : 0;
}

int d3d_op_time_table(d3d_handle* h, const float* t_host, int32_t R, float* out, void* stream) {
  if (!h || !t_host || !out) return -1;
  if (!h->cfg.with_time_emb) return fail(h, -3, "handle was created with with_time_emb = 0");
  if (R < 1 || R > h->t_rows_cap) return fail(h, -2, "R out of range");
  int r = check_weights(h);
  if (r) return r;
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CK(cudaMemcpyAsync(h->t_f32, t_host, sizeof(float) * R, cudaMemcpyHostToDevice, st));
  CK(cudaStreamSynchronize(st));
  return compute_time_table(h, h->t_f32, R, out, st);
}

}  // extern "C"

namespace {
struct OpLinearBufs {
  OperandBuf a;
  Lin w;
  __half *o_hi = nullptr, *o_lo = nullptr;
  uint8_t* o_sf = nullptr;
  std::vector<void*> mine;
  ~OpLinearBufs() { for (void* p : mine) cudaFree(p); }
};
template <typename T>
cudaError_t tmp_alloc(OpLinearBufs& b, T** p, int64_t n) {
  void* q = nullptr;
  cudaError_t e = cudaMalloc(&q, static_cast<size_t>(n) * sizeof(T));
  if (e != cudaSuccess) return e;
  e = cudaMemset(q, 0, static_cast<size_t>(n) * sizeof(T));
  b.mine.push_back(q);
  *p = static_cast<T*>(q);
  return e;
}
int prep_op_linear(d3d_handle* h, OpLinearBufs& b, int64_t M, int N, int K, int act, int fmt) {
  const int64_t Mp = (M + 511) / 512 * 512;
  CK(tmp_alloc(b, &b.a.hi, Mp * K));
  CK(tmp_alloc(b, &b.a.lo, Mp * K));
  CK(tmp_alloc(b, &b.w.hi, static_cast<int64_t>(N) * K));
  CK(tmp_alloc(b, &b.w.lo, static_cast<int64_t>(N) * K));
  b.w.N = N;
  b.w.K = K;
  if (act) {
    CK(tmp_alloc(b, &b.o_hi, Mp * N));
    CK(tmp_alloc(b, &b.o_lo, Mp * N));
    if (fmt == FMT_F4C) b.o_sf = reinterpret_cast<uint8_t*>(b.o_lo) + op_sf_base(Mp, N);
  }
  if (make_maps(&b.a.m_hi, &b.a.m_lo, b.a.hi, b.a.lo, Mp, K, fmt) || make_maps(&b.w.m_hi, &b.w.m_lo, b.w.hi, b.w.lo, N, K, fmt) ||
      make_maps(&b.w.m_hi64, &b.w.m_lo64, b.w.hi, b.w.lo, N, K, fmt, 64) || make_sf(&b.a.sf, &b.a.m_sf, b.a.lo, Mp, K, fmt) ||
      make_sf(&b.w.sf, &b.w.m_sf, b.w.lo, N, K, fmt))
    return fail(h, -20, "cuTensorMapEncodeTiled failed");
  return 0;
}
}  // namespace

extern "C" {

int d3d_op_linear(d3d_handle* h, const float* a, const float* w, const float* bias, const float* residual, float* out,
                  int64_t M, int32_t N, int32_t K, int32_t act, int32_t gemm_mode, void* stream) {
  if (!h || !a || !w || !bias || !out) return -1;
  if (M < 1 || N % 128 != 0 || K % 64 != 0 || N < 128 || K < 64) return fail(h, -2, "need M>=1, N%128==0, K%64==0");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  OpLinearBufs b;
  const int fmt = mode_fmt(gemm_mode);
  int r = prep_op_linear(h, b, M, N, K, act, fmt);
  if (r) return r;
  b.w.bias = const_cast<float*>(bias);
  if (fmt == FMT_F4C && (N % 256 != 0 || K % 128 != 0)) return fail(h, -2, "the F4C GEMM needs N%256==0 and K%128==0");
  KL(launch_split(a, b.a.hi, b.a.lo, b.a.sf, M, K, fmt, 0, st));
  KL(launch_split(w, b.w.hi, b.w.lo, b.w.sf, N, K, fmt, 1, st));
  if (act) {
    if ((r = run_gemm(h, b.a, b.w, M, EPI_GELU_SPLIT, nullptr, nullptr, b.o_hi, b.o_lo, nullptr, gemm_mode, st, nullptr, b.o_sf))) return r;
    KL(launch_merge(b.o_hi, b.o_lo, b.o_sf, out, M, N, fmt, st));
  } else if (residual && gemm_mode == D3D_GEMM_TC_F4C && N % 256 == 0 && env_int("D3D_GEMM_RED", 1) == 1) {
    // as the sampler runs proj / fc2: the residual already sits in `out`, the epilogue reduce-adds into it
    CUtensorMap om;
    if (make_f32_tile_map(&om, out, M, N)) return fail(h, -20, "cuTensorMapEncodeTiled failed");
    CK(cudaMemcpyAsync(out, residual, static_cast<size_t>(M) * N * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if ((r = run_gemm(h, b.a, b.w, M, EPI_F32, out, out, nullptr, nullptr, nullptr, gemm_mode, st, nullptr, nullptr, nullptr, &om))) return r;
  } else {
    if ((r = run_gemm(h, b.a, b.w, M, EPI_F32, residual, out, nullptr, nullptr, nullptr, gemm_mode, st))) return r;
  }
  CK(cudaStreamSynchronize(st));
  return 0;
}

int d3d_op_linear_ln(d3d_handle* h, const float* a, const float* w, const float* bias, const float* residual,
                     const float* gamma, const float* beta, float eps, float* x_out, float* ln_out, int64_t M, int32_t K,
                     void* stream) {
  if (!h || !a || !w || !bias || !residual || !gamma || !beta || !x_out || !ln_out) return -1;
  if (M < 1 || K % 64 != 0 || K < 64) return fail(h, -2, "need M>=1, K%64==0");
  if (!can_fuse_ln(h, D3D_GEMM_TC_F8C)) return fail(h, -3, "the fused GEMM + LayerNorm epilogue needs the F8C CTA-pair kernel");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  OpLinearBufs b;
  int r = prep_op_linear(h, b, M, kC, K, 1 /*allocates o_hi / o_lo [M, 512]*/, FMT_F8C);
  if (r) return r;
  b.w.bias = const_cast<float*>(bias);
  KL(launch_split(a, b.a.hi, b.a.lo, nullptr, M, K, FMT_F8C, 0, st));
  KL(launch_split(w, b.w.hi, b.w.lo, nullptr, kC, K, FMT_F8C, 1, st));
  OperandBuf dst;
  dst.hi = b.o_hi;
  dst.lo = b.o_lo;
  const LnFuse ln{gamma, beta, eps, &dst};
  if ((r = run_gemm(h, b.a, b.w, M, EPI_F32, residual, x_out, nullptr, nullptr, nullptr, D3D_GEMM_TC_F8C, st, &ln))) return r;
  KL(launch_merge(b.o_hi, b.o_lo, nullptr, ln_out, M, kC, FMT_F8C, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}

int d3d_op_linear_dln_linear(d3d_handle* h, const float* a, const float* w, const float* bias, const float* residual,
                             const float* gamma, const float* beta, float eps, const float* w2, const float* b2,
                             float* x_out, float* hid_out, int64_t M, int32_t K, void* stream) {
  if (!h || !a || !w || !bias || !residual || !gamma || !beta || !w2 || !b2 || !x_out || !hid_out) return -1;
  if (M < 1 || K % 128 != 0 || K < 128) return fail(h, -2, "need M>=1, K%128==0");
  if (pick_cg(kC) != 2) return fail(h, -3, "the deferred-LayerNorm epilogues need the CTA-pair kernel");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  OpLinearBufs b1, b2b;
  int r = prep_op_linear(h, b1, M, kC, K, 1 /*o_hi / o_lo [M,512]: the emitted operand*/, FMT_F4C);
  if (r) return r;
  if ((r = prep_op_linear(h, b2b, M, kHidden, kC, 1, FMT_F4C))) return r;
  const int64_t Mp = (M + 511) / 512 * 512;
  float2* stats = nullptr;
  float *wfold = nullptr, *colsum = nullptr, *cbias = nullptr;
  CK(tmp_alloc(b1, &stats, 8 * Mp));
  CK(tmp_alloc(b1, &wfold, static_cast<int64_t>(kHidden) * kC));
  CK(tmp_alloc(b1, &colsum, kHidden));
  CK(tmp_alloc(b1, &cbias, kHidden));
  b1.w.bias = const_cast<float*>(bias);
  b2b.w.bias = const_cast<float*>(b2);
  KL(launch_split(a, b1.a.hi, b1.a.lo, b1.a.sf, M, K, FMT_F4C, 0, st));
  KL(launch_split(w, b1.w.hi, b1.w.lo, b1.w.sf, kC, K, FMT_F4C, 1, st));
  KL(launch_fold_ln_linear(w2, gamma, beta, b2, wfold, colsum, cbias, kHidden, kC, st));
  KL(launch_split(wfold, b2b.w.hi, b2b.w.lo, b2b.w.sf, kHidden, kC, FMT_F4C, 1, st));
  CK(cudaMemcpyAsync(x_out, residual, static_cast<size_t>(M) * kC * sizeof(float), cudaMemcpyDeviceToDevice, st));
  // the emitted operand of the first GEMM IS the A operand of the second: give it the second one's tensor maps
  OperandBuf mid = b2b.a;
  const DeferLn dl{&mid, stats, colsum, cbias, eps};
  if ((r = run_gemm(h, b1.a, b1.w, M, EPI_F32_EMIT, x_out, x_out, nullptr, nullptr, nullptr, D3D_GEMM_TC_F4C, st, nullptr, nullptr, &dl))) return r;
  if ((r = run_gemm(h, mid, b2b.w, M, EPI_GELU_DLN, nullptr, nullptr, b2b.o_hi, b2b.o_lo, nullptr, D3D_GEMM_TC_F4C, st, nullptr, b2b.o_sf, &dl))) return r;
  KL(launch_merge(b2b.o_hi, b2b.o_lo, b2b.o_sf, hid_out, M, kHidden, FMT_F4C, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}

int d3d_op_linear_bench(d3d_handle* h, int64_t M, int32_t N, int32_t K, int32_t act, int32_t gemm_mode, int32_t iters,
                        float* ms_per_launch) {
  if (!h || !ms_per_launch || iters < 1) return -1;
  if (M < 1 || N % 128 != 0 || K % 64 != 0) return fail(h, -2, "need M>=1, N%128==0, K%64==0");
  DeviceGuard guard(h->cfg.device);
  cudaStream_t st = h->cap_stream;
  OpLinearBufs b;
  const int fmt = mode_fmt(gemm_mode);
  // act: 0 fp32 out, 1 GELU -> operand, 2 fp32 out + in-place residual, 3 = 2 + emitted operand + row statistics
  // (EPI_F32_EMIT), 4 GELU with the deferred LayerNorm (EPI_GELU_DLN)
  if (act < 0 || act > 4) return fail(h, -2, "act out of range");
  if (act >= 3 && gemm_mode != D3D_GEMM_TC_F4C) return fail(h, -3, "act 3 / 4 need D3D_GEMM_TC_F4C");
  int r = prep_op_linear(h, b, M, N, K, act == 2 ? 0 : act, fmt);
  if (r) return r;
  const int64_t Mp = (M + 511) / 512 * 512;
  float2* stats = nullptr;
  float* colsum = nullptr;
  OperandBuf emit;
  if (act >= 3) {
    CK(tmp_alloc(b, &stats, 8 * Mp));
    CK(tmp_alloc(b, &colsum, N));
    emit.hi = b.o_hi; emit.lo = b.o_lo; emit.sf = b.o_sf;
  }
  float *fa = nullptr, *fo = nullptr, *fb = nullptr;
  CK(tmp_alloc(b, &fa, M * K > static_cast<int64_t>(N) * K ? M * K : static_cast<int64_t>(N) * K));
  CK(tmp_alloc(b, &fo, M * N));
  CK(tmp_alloc(b, &fb, N));
  b.w.bias = fb;
  // deterministic non-trivial operands: a 0.01-step ramp pattern split into halves
  std::vector<float> host(1 << 20);
  for (size_t i = 0; i < host.size(); ++i) host[i] = static_cast<float>(static_cast<int>((i * 2654435761u) >> 20 & 1023) - 512) * (1.0f / 512.0f);
  const int64_t na = M * K;
  for (int64_t off = 0; off < na; off += static_cast<int64_t>(host.size()))
    CK(cudaMemcpy(fa + off, host.data(), sizeof(float) * static_cast<size_t>(std::min<int64_t>(host.size(), na - off)), cudaMemcpyHostToDevice));
  CK(launch_split(fa, b.a.hi, b.a.lo, b.a.sf, M, K, fmt, 0, st));
  CK(launch_split(fa, b.w.hi, b.w.lo, b.w.sf, N, K, fmt, 1, st));
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  const DeferLn dl{&emit, stats, colsum, fb, 1e-6f};
  CUtensorMap fo_map;
  if (make_f32_tile_map(&fo_map, fo, M, N)) return fail(h, -20, "cuTensorMapEncodeTiled failed");
  auto once = [&]() -> int {
    if (act == 1) return run_gemm(h, b.a, b.w, M, EPI_GELU_SPLIT, nullptr, nullptr, b.o_hi, b.o_lo, nullptr, gemm_mode, st, nullptr, b.o_sf);
    if (act == 2) return run_gemm(h, b.a, b.w, M, EPI_F32, fo, fo, nullptr, nullptr, nullptr, gemm_mode, st, nullptr, nullptr, nullptr, &fo_map);
    if (act == 3) return run_gemm(h, b.a, b.w, M, EPI_F32_EMIT, fo, fo, nullptr, nullptr, nullptr, gemm_mode, st, nullptr, nullptr, &dl);
    if (act == 4) return run_gemm(h, b.a, b.w, M, EPI_GELU_DLN, nullptr, nullptr, b.o_hi, b.o_lo, nullptr, gemm_mode, st, nullptr, b.o_sf, &dl);
    return run_gemm(h, b.a, b.w, M, EPI_F32, nullptr, fo, nullptr, nullptr, nullptr, gemm_mode, st);
  };
  for (int i = 0; i < 3; ++i)
    if ((r = once())) return r;
  CK(cudaEventRecord(e0, st));
  for (int i = 0; i < iters; ++i)
    if ((r = once())) return r;
  CK(cudaEventRecord(e1, st));
  CK(cudaStreamSynchronize(st));
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *ms_per_launch = ms / iters;
  return 0;
}

}  // extern "C"
