// Row-wise (memory-bound) kernels: one warp owns one C-wide token row (C = 512 or 256, a template parameter), lane l holds
// columns {128*i + 4*l .. +3 : i < C / 128} -- N = C / 32 values per lane -- so every global access is a fully coalesced
// 128-bit transaction.
//
//   lift_ln            G-lift : fusion_layer (K=5) + Spatial_pos_embed + block-0 time vector + norm1   (MODEL:250,230-233,113-116,127)
//   postnorm_add_ln    G-ln   : Spatial_/Temporal_norm + Temporal_pos_embed + next block's time vector + next norm1
//   ln_split           G-ln   : norm2 -> split fp16 A operand of fc1                                  (MODEL:128)
//   head_ddim          G-head+ddim : Temporal_norm + head LayerNorm(1e-5) + Linear(C->3) + clamp + DDIM update
//                                                                                  (MODEL:245,255; DIFF:256,283-297)
//   tta_merge, mpjpe   G-tta  : RUN:583-588, LOSS:15-27
#include <cstdlib>
#include "kernels.cuh"
#include "operand.cuh"
#include "ptx.cuh"

namespace d3d {
namespace {

constexpr int kWarpsPerCta = 8;
// the two-row kernels are capped at 64 registers (4 CTAs = 32 warps per SM instead of 24): LayerNorm class 498 -> 480 ms per
// cfg3 step (profiles/r02y3_*); D3D_ROWS2_MIN_CTAS=1 builds the uncapped forms
#ifndef D3D_ROWS2_MIN_CTAS
#define D3D_ROWS2_MIN_CTAS 4
#endif

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int N>
__device__ __forceinline__ void load_row(const float* __restrict__ p, int lane, float (&v)[N]) {
#pragma unroll
  for (int i = 0; i < N / 4; ++i) {
    const float4 t = *reinterpret_cast<const float4*>(p + 128 * i + 4 * lane);
    v[4 * i + 0] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
  }
}
template <int N>
__device__ __forceinline__ void load_row_ldg(const float* __restrict__ p, int lane, float (&v)[N]) {
#pragma unroll
  for (int i = 0; i < N / 4; ++i) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p + 128 * i + 4 * lane));
    v[4 * i + 0] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
  }
}
template <int N>
__device__ __forceinline__ void store_row(float* __restrict__ p, int lane, const float (&v)[N]) {
#pragma unroll
  for (int i = 0; i < N / 4; ++i)
    *reinterpret_cast<float4*>(p + 128 * i + 4 * lane) = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
}
// a += b  /  a += s * b  over the lane's N columns, as N / 2 packed pairs
template <int N>
__device__ __forceinline__ void add16(float (&a)[N], const float (&b)[N]) {
#pragma unroll
  for (int i = 0; i < N / 2; ++i)
    ptx::unpack2(ptx::add2(ptx::pack2(a[2 * i], a[2 * i + 1]), ptx::pack2(b[2 * i], b[2 * i + 1])), a[2 * i], a[2 * i + 1]);
}
template <int N>
__device__ __forceinline__ void fma16(float (&a)[N], float s, const float (&b)[N]) {
  const ptx::f32x2 s2 = ptx::splat2(s);
#pragma unroll
  for (int i = 0; i < N / 2; ++i)
    ptx::unpack2(ptx::fma2(s2, ptx::pack2(b[2 * i], b[2 * i + 1]), ptx::pack2(a[2 * i], a[2 * i + 1])), a[2 * i], a[2 * i + 1]);
}

// GEMM A operand of token row `row` (K = C = 32 N) in the handle's operand format (operand.cuh); `second` / `sf` are the
// BASE pointers of the operand's second array and (FMT_F4C) its scale-factor array.
template <int FMT, int N>
__device__ __forceinline__ void store_operand(__half* __restrict__ hi, __half* __restrict__ second,
                                              uint8_t* __restrict__ sf, int64_t row, int lane, const float (&v)[N]) {
  constexpr int kC = 32 * N;
  if (FMT != FMT_F4C) {
#pragma unroll
    for (int i = 0; i < N / 4; ++i) {
      const float x[4] = {v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]};
      op_store4<FMT>(hi + row * kC, second + row * kC, kC, 128 * i + 4 * lane, x);
    }
    return;
  }
  // FMT_F4C: the lane's 4 columns of chunk i belong to the 32-column block (4 i + lane / 8).  The scale byte is a
  // monotone function of the block maximum, so the 8 lanes of a block reduce the two BYTES (P: q4(x), k-blocks 0..15;
  // Q: q4(x - hi), k-blocks C/32 .. C/16 - 1) packed in one register with three shuffles + packed-halfword maxima.
  uint8_t* c4 = reinterpret_cast<uint8_t*>(second) + row * kC;
  __half* hrow = hi + row * kC;
  // scale bytes of (row, k-block 4 i + g) sit at sf_row + 512 i + g (P) and sf_row + 512 (C / 128 + i) + g (Q)
  uint8_t* sf_row = sf + (static_cast<size_t>(row >> 7) * (kC / 64)) * 512 + 16 * (row & 31) + 4 * ((row & 127) >> 5) + (lane >> 3);
#pragma unroll
  for (int i = 0; i < N / 4; ++i) {
    float x[4], l[4];
    const __half2 h01 = __floats2half2_rn(v[4 * i], v[4 * i + 1]), h23 = __floats2half2_rn(v[4 * i + 2], v[4 * i + 3]);
    const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
    const ptx::f32x2 x01 = ptx::pack2(v[4 * i], v[4 * i + 1]), x23 = ptx::pack2(v[4 * i + 2], v[4 * i + 3]);
    const ptx::f32x2 l01 = ptx::sub2(x01, ptx::pack2(f01.x, f01.y)), l23 = ptx::sub2(x23, ptx::pack2(f23.x, f23.y));
    ptx::unpack2(l01, l[0], l[1]);
    ptx::unpack2(l23, l[2], l[3]);
    const float ax = fmaxf(fmaxf(fabsf(v[4 * i]), fabsf(v[4 * i + 1])), fmaxf(fabsf(v[4 * i + 2]), fabsf(v[4 * i + 3])));
    const float al = fmaxf(fmaxf(fabsf(l[0]), fabsf(l[1])), fmaxf(fabsf(l[2]), fabsf(l[3])));
    uint32_t bb = op_ue8m0_of(ax) | (op_ue8m0_of(al) << 16);
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) bb = __vmaxu2(bb, __shfl_xor_sync(0xffffffffu, bb, o));
    const uint32_t bp = bb & 0xffu, bq = bb >> 16;
    const ptx::f32x2 ip = ptx::splat2(op_ue8m0_inv(bp)), iq = ptx::splat2(op_ue8m0_inv(bq));
    const int col = 128 * i + 4 * lane;
    *reinterpret_cast<uint2*>(hrow + col) =
        make_uint2(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23));
    ptx::unpack2(ptx::mul2(x01, ip), x[0], x[1]);
    ptx::unpack2(ptx::mul2(x23, ip), x[2], x[3]);
    *reinterpret_cast<uint16_t*>(c4 + (col >> 1)) = static_cast<uint16_t>(op_e2m1x2(x[0], x[1]) | (op_e2m1x2(x[2], x[3]) << 8));
    ptx::unpack2(ptx::mul2(l01, iq), l[0], l[1]);
    ptx::unpack2(ptx::mul2(l23, iq), l[2], l[3]);
    *reinterpret_cast<uint16_t*>(c4 + (kC >> 1) + (col >> 1)) =
        static_cast<uint16_t>(op_e2m1x2(l[0], l[1]) | (op_e2m1x2(l[2], l[3]) << 8));
    if ((lane & 7) == 0) {       // lanes 0, 8, 16, 24: four adjacent bytes of one scale-factor atom
      sf_row[512 * i] = static_cast<uint8_t>(bp);
      sf_row[512 * (N / 4 + i)] = static_cast<uint8_t>(bq);
    }
  }
}

// y = (x - mean) * rstd * gamma + beta over the C columns held by the warp (two-pass variance in registers).  The
// element-wise work runs on packed fp32 pairs (FADD2 / FFMA2 / FMUL2: two IEEE-rn operations per issue slot): with the
// block-scaled operand format these kernels are bound by instruction issue, not by HBM.
template <int N>
__device__ __forceinline__ float ln_center(const float (&x)[N], ptx::f32x2 (&xp)[N / 2]);
__device__ __forceinline__ ptx::f32x2 ln_rstd(float var, float eps);
template <int N>
__device__ __forceinline__ void layernorm_row(const float (&x)[N], const float* __restrict__ gamma,
                                              const float* __restrict__ beta, float eps, int lane, float (&y)[N]) {
  ptx::f32x2 xp[N / 2];
  const float var = ln_center(x, xp);
  // 1 / sqrt(var + eps): MUFU.RSQ + one Newton step (< 1 ulp) -- the IEEE sqrt + division pair cost ~25 instructions with
  // its slow-path calls (ln_rstd)
  const ptx::f32x2 rstd = ln_rstd(var, eps);
#pragma unroll
  for (int i = 0; i < N / 4; ++i) {
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + 128 * i + 4 * lane));
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta + 128 * i + 4 * lane));
    ptx::unpack2(ptx::fma2(ptx::mul2(xp[2 * i], rstd), ptx::pack2(g.x, g.y), ptx::pack2(b.x, b.y)), y[4 * i], y[4 * i + 1]);
    ptx::unpack2(ptx::fma2(ptx::mul2(xp[2 * i + 1], rstd), ptx::pack2(g.z, g.w), ptx::pack2(b.z, b.w)), y[4 * i + 2], y[4 * i + 3]);
  }
}

// The same LayerNorm on TWO rows of one warp (rows t, t + 1), every parameter vector loaded ONCE for both.  ncu on the
// one-row kernels (profiles/r02n_full_*.md, r02f_full_postnorm_add_ln.md): l1tex throughput 77-95 % -- each row re-read
// 2 KB per parameter vector through L1 (24 of postnorm's 36 memory instructions), and at the step's power-capped clock
// that, not HBM, set their time.  Per-row arithmetic is identical to layernorm_row (results do not depend on the partner).
template <int N>
__device__ __forceinline__ float ln_center(const float (&x)[N], ptx::f32x2 (&xp)[N / 2]) {      // xp = x - mean; returns var
  static_assert(N == 8 || N == 16, "C = 256 or 512");
  constexpr int kC = 32 * N;
#pragma unroll
  for (int i = 0; i < N / 2; ++i) xp[i] = ptx::pack2(x[2 * i], x[2 * i + 1]);
  ptx::f32x2 sp;
  if constexpr (N == 16)
    sp = ptx::add2(ptx::add2(ptx::add2(xp[0], xp[1]), ptx::add2(xp[2], xp[3])),
                   ptx::add2(ptx::add2(xp[4], xp[5]), ptx::add2(xp[6], xp[7])));
  else
    sp = ptx::add2(ptx::add2(xp[0], xp[1]), ptx::add2(xp[2], xp[3]));
  float s0, s1;
  ptx::unpack2(sp, s0, s1);
  const float mean = warp_sum(s0 + s1) * (1.0f / kC);
  const ptx::f32x2 nm = ptx::splat2(-mean);
  ptx::f32x2 qp = ptx::splat2(0.f);
#pragma unroll
  for (int i = 0; i < N / 2; ++i) {
    xp[i] = ptx::add2(xp[i], nm);
    qp = ptx::fma2(xp[i], xp[i], qp);
  }
  ptx::unpack2(qp, s0, s1);
  return warp_sum(s0 + s1) * (1.0f / kC);
}
__device__ __forceinline__ ptx::f32x2 ln_rstd(float var, float eps) {
  const float ve = var + eps;
  float r0;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r0) : "f"(ve));
  return ptx::splat2(r0 * fmaf(-0.5f * ve, r0 * r0, 1.5f));
}
// y_r = LN(x_r) (+ add) for r = 0, 1; `add` (optional, a C-vector common to both rows) is added after beta
template <int N>
__device__ __forceinline__ void layernorm_2rows(const float (&x0)[N], const float (&x1)[N], const float* __restrict__ gamma,
                                                const float* __restrict__ beta, const float* __restrict__ add, float eps,
                                                int lane, float (&y0)[N], float (&y1)[N]) {
  ptx::f32x2 p0[N / 2], p1[N / 2];
  const float v0 = ln_center(x0, p0), v1 = ln_center(x1, p1);
  const ptx::f32x2 r0 = ln_rstd(v0, eps), r1 = ln_rstd(v1, eps);
#pragma unroll
  for (int i = 0; i < N / 4; ++i) {
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + 128 * i + 4 * lane));
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta + 128 * i + 4 * lane));
    const ptx::f32x2 g01 = ptx::pack2(g.x, g.y), g23 = ptx::pack2(g.z, g.w), b01 = ptx::pack2(b.x, b.y), b23 = ptx::pack2(b.z, b.w);
    ptx::f32x2 a0 = ptx::fma2(ptx::mul2(p0[2 * i], r0), g01, b01), a1 = ptx::fma2(ptx::mul2(p0[2 * i + 1], r0), g23, b23);
    ptx::f32x2 c0 = ptx::fma2(ptx::mul2(p1[2 * i], r1), g01, b01), c1 = ptx::fma2(ptx::mul2(p1[2 * i + 1], r1), g23, b23);
    if (add) {
      const float4 w = __ldg(reinterpret_cast<const float4*>(add + 128 * i + 4 * lane));
      const ptx::f32x2 w01 = ptx::pack2(w.x, w.y), w23 = ptx::pack2(w.z, w.w);
      a0 = ptx::add2(a0, w01); a1 = ptx::add2(a1, w23);
      c0 = ptx::add2(c0, w01); c1 = ptx::add2(c1, w23);
    }
    ptx::unpack2(a0, y0[4 * i], y0[4 * i + 1]);
    ptx::unpack2(a1, y0[4 * i + 2], y0[4 * i + 3]);
    ptx::unpack2(c0, y1[4 * i], y1[4 * i + 1]);
    ptx::unpack2(c1, y1[4 * i + 2], y1[4 * i + 3]);
  }
}

template <int C, int FMT>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
lift_ln_kernel(const float* __restrict__ x2d, const float* __restrict__ y3, const float* __restrict__ x5,
               const float* __restrict__ wf_t, const float* __restrict__ bf, const float* __restrict__ spos,
               const float* __restrict__ tvec, int64_t tvec_stride, LnParams ln1, float* __restrict__ X,
               __half* __restrict__ a_hi, __half* __restrict__ a_lo, uint8_t* __restrict__ a_sf, int64_t T, int J,
               int tokens_per_clip) {
  const int lane = threadIdx.x & 31;
  const int64_t t = static_cast<int64_t>(blockIdx.x) * kWarpsPerCta + (threadIdx.x >> 5);
  if (t >= T) return;
  float in[5];
  if (x5) {
#pragma unroll
    for (int k = 0; k < 5; ++k) in[k] = __ldg(x5 + t * 5 + k);
  } else {
    in[0] = __ldg(x2d + t * 2); in[1] = __ldg(x2d + t * 2 + 1);
    in[2] = __ldg(y3 + t * 3); in[3] = __ldg(y3 + t * 3 + 1); in[4] = __ldg(y3 + t * 3 + 2);
  }
  float v[C / 32], w[C / 32];
  // F.linear: sum_k in_k * W[c][k] + b[c]
#pragma unroll
  for (int i = 0; i < C / 32; ++i) v[i] = 0.f;
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    load_row_ldg(wf_t + k * C, lane, w);
    fma16(v, in[k], w);
  }
  load_row_ldg(bf, lane, w);
  add16(v, w);
  // token indices fit 32 bits (launchers check T < 2^31): 32-bit divisions instead of the 64-bit software routine,
  // which cost these issue-bound kernels ~100 instructions per row
  const uint32_t t32 = static_cast<uint32_t>(t);
  load_row_ldg(spos + static_cast<size_t>(t32 % static_cast<uint32_t>(J)) * C, lane, w);
  add16(v, w);
  if (tvec) {
    const float* tv = tvec;
    if (tvec_stride != 0) tv += static_cast<int64_t>(t32 / static_cast<uint32_t>(tokens_per_clip)) * tvec_stride;
    load_row_ldg(tv, lane, w);
    add16(v, w);
  }
  store_row(X + t * C, lane, v);
  float a[C / 32];
  layernorm_row(v, ln1.gamma, ln1.beta, 1e-6f, lane, a);
  store_operand<FMT>(a_hi, a_lo, a_sf, t, lane, a);
}

// lift_ln on two rows per warp: the five fusion_layer weight rows, its bias, the time vector and the norm1 parameters are
// loaded once for both tokens (only the Spatial_pos_embed row differs); eval only (one time vector for every clip).
template <int C, int FMT>
__global__ void __launch_bounds__(kWarpsPerCta * 32, D3D_ROWS2_MIN_CTAS)
lift_ln2_kernel(const float* __restrict__ x2d, const float* __restrict__ y3, const float* __restrict__ x5,
                const float* __restrict__ wf_t, const float* __restrict__ bf, const float* __restrict__ spos,
                const float* __restrict__ tvec, LnParams ln1, float* __restrict__ X, __half* __restrict__ a_hi,
                __half* __restrict__ a_lo, uint8_t* __restrict__ a_sf, int64_t T, int J) {
  const int lane = threadIdx.x & 31;
  const int64_t t = (static_cast<int64_t>(blockIdx.x) * kWarpsPerCta + (threadIdx.x >> 5)) * 2;
  if (t >= T) return;
  const bool two = t + 1 < T;
  const int64_t t1 = two ? t + 1 : t;
  float in0[5], in1[5];
  if (x5) {
#pragma unroll
    for (int k = 0; k < 5; ++k) { in0[k] = __ldg(x5 + t * 5 + k); in1[k] = __ldg(x5 + t1 * 5 + k); }
  } else {
    in0[0] = __ldg(x2d + t * 2); in0[1] = __ldg(x2d + t * 2 + 1);
    in0[2] = __ldg(y3 + t * 3); in0[3] = __ldg(y3 + t * 3 + 1); in0[4] = __ldg(y3 + t * 3 + 2);
    in1[0] = __ldg(x2d + t1 * 2); in1[1] = __ldg(x2d + t1 * 2 + 1);
    in1[2] = __ldg(y3 + t1 * 3); in1[3] = __ldg(y3 + t1 * 3 + 1); in1[4] = __ldg(y3 + t1 * 3 + 2);
  }
  float v0[C / 32], v1[C / 32], w[C / 32];
#pragma unroll
  for (int i = 0; i < C / 32; ++i) { v0[i] = 0.f; v1[i] = 0.f; }
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    load_row_ldg(wf_t + k * C, lane, w);
    fma16(v0, in0[k], w);
    fma16(v1, in1[k], w);
  }
  load_row_ldg(bf, lane, w);
  add16(v0, w);
  add16(v1, w);
  const uint32_t j0 = static_cast<uint32_t>(t) % static_cast<uint32_t>(J);
  const uint32_t j1 = j0 + 1 == static_cast<uint32_t>(J) ? 0u : j0 + 1;
  load_row_ldg(spos + static_cast<size_t>(j0) * C, lane, w);
  add16(v0, w);
  load_row_ldg(spos + static_cast<size_t>(j1) * C, lane, w);
  add16(v1, w);
  if (tvec) {
    load_row_ldg(tvec, lane, w);
    add16(v0, w);
    add16(v1, w);
  }
  store_row(X + t * C, lane, v0);
  if (two) store_row(X + (t + 1) * C, lane, v1);
  float a0[C / 32], a1[C / 32];
  layernorm_2rows(v0, v1, ln1.gamma, ln1.beta, nullptr, 1e-6f, lane, a0, a1);
  store_operand<FMT>(a_hi, a_lo, a_sf, t, lane, a0);
  if (two) store_operand<FMT>(a_hi, a_lo, a_sf, t + 1, lane, a1);
}

template <int C, int FMT>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
postnorm_add_ln_kernel(float* __restrict__ X, LnParams post, const float* __restrict__ tpos,
                       const float* __restrict__ tvec, int64_t tvec_stride, LnParams ln1, __half* __restrict__ a_hi,
                       __half* __restrict__ a_lo, uint8_t* __restrict__ a_sf, int64_t T, int J, int F) {
  const int lane = threadIdx.x & 31;
  const int64_t t = static_cast<int64_t>(blockIdx.x) * kWarpsPerCta + (threadIdx.x >> 5);
  if (t >= T) return;
  float x[C / 32], z[C / 32], w[C / 32];
  load_row(X + t * C, lane, x);
  layernorm_row(x, post.gamma, post.beta, 1e-6f, lane, z);
  if (tpos) {
    load_row_ldg(tpos + static_cast<size_t>((static_cast<uint32_t>(t) / static_cast<uint32_t>(J)) % static_cast<uint32_t>(F)) * C, lane, w);
    add16(z, w);
  }
  if (tvec) {          // eval: every clip shares t (tvec_stride == 0), no clip index needed
    const float* tv = tvec;
    if (tvec_stride != 0) tv += static_cast<int64_t>(static_cast<uint32_t>(t) / static_cast<uint32_t>(J * F)) * tvec_stride;
    load_row_ldg(tv, lane, w);
    add16(z, w);
  }
  store_row(X + t * C, lane, z);
  layernorm_row(z, ln1.gamma, ln1.beta, 1e-6f, lane, x);
  store_operand<FMT>(a_hi, a_lo, a_sf, t, lane, x);
}

template <int C, int FMT>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
ln_split_kernel(const float* __restrict__ X, LnParams ln, float eps, __half* __restrict__ a_hi,
                __half* __restrict__ a_lo, uint8_t* __restrict__ a_sf, int64_t T) {
  const int lane = threadIdx.x & 31;
  const int64_t t = static_cast<int64_t>(blockIdx.x) * kWarpsPerCta + (threadIdx.x >> 5);
  if (t >= T) return;
  float x[C / 32], y[C / 32];
  load_row(X + t * C, lane, x);
  layernorm_row(x, ln.gamma, ln.beta, eps, lane, y);
  store_operand<FMT>(a_hi, a_lo, a_sf, t, lane, y);
}

// Two rows per warp (rows 2 w, 2 w + 1 of the launch): the production forms of ln_split / postnorm_add_ln when no
// per-row additive term is needed (eval: one time vector for every clip; Temporal_pos_embed only after block 0).
template <int C, int FMT>
__global__ void __launch_bounds__(kWarpsPerCta * 32, D3D_ROWS2_MIN_CTAS)
ln_split2_kernel(const float* __restrict__ X, LnParams ln, float eps, __half* __restrict__ a_hi, __half* __restrict__ a_lo,
                 uint8_t* __restrict__ a_sf, int64_t T) {
  const int lane = threadIdx.x & 31;
  const int64_t t = (static_cast<int64_t>(blockIdx.x) * kWarpsPerCta + (threadIdx.x >> 5)) * 2;
  if (t >= T) return;
  const bool two = t + 1 < T;
  float x0[C / 32], x1[C / 32], y0[C / 32], y1[C / 32];
  load_row(X + t * C, lane, x0);
  load_row(X + (two ? t + 1 : t) * C, lane, x1);
  layernorm_2rows(x0, x1, ln.gamma, ln.beta, nullptr, eps, lane, y0, y1);
  store_operand<FMT>(a_hi, a_lo, a_sf, t, lane, y0);
  if (two) store_operand<FMT>(a_hi, a_lo, a_sf, t + 1, lane, y1);
}

template <int C, int FMT>
__global__ void __launch_bounds__(kWarpsPerCta * 32, D3D_ROWS2_MIN_CTAS)
postnorm_add_ln2_kernel(float* __restrict__ X, LnParams post, const float* __restrict__ tvec, LnParams ln1,
                        __half* __restrict__ a_hi, __half* __restrict__ a_lo, uint8_t* __restrict__ a_sf, int64_t T) {
  const int lane = threadIdx.x & 31;
  const int64_t t = (static_cast<int64_t>(blockIdx.x) * kWarpsPerCta + (threadIdx.x >> 5)) * 2;
  if (t >= T) return;
  const bool two = t + 1 < T;
  float x0[C / 32], x1[C / 32], z0[C / 32], z1[C / 32];
  load_row(X + t * C, lane, x0);
  load_row(X + (two ? t + 1 : t) * C, lane, x1);
  layernorm_2rows(x0, x1, post.gamma, post.beta, tvec, 1e-6f, lane, z0, z1);
  store_row(X + t * C, lane, z0);
  if (two) store_row(X + (t + 1) * C, lane, z1);
  layernorm_2rows(z0, z1, ln1.gamma, ln1.beta, nullptr, 1e-6f, lane, x0, x1);
  store_operand<FMT>(a_hi, a_lo, a_sf, t, lane, x0);
  if (two) store_operand<FMT>(a_hi, a_lo, a_sf, t + 1, lane, x1);
}

template <int C>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
ln_f32_kernel(const float* __restrict__ X, LnParams ln, float eps, float* __restrict__ out, int64_t T) {
  const int lane = threadIdx.x & 31;
  const int64_t t = static_cast<int64_t>(blockIdx.x) * kWarpsPerCta + (threadIdx.x >> 5);
  if (t >= T) return;
  float x[C / 32], y[C / 32];
  load_row(X + t * C, lane, x);
  layernorm_row(x, ln.gamma, ln.beta, eps, lane, y);
  store_row(out + t * C, lane, y);
}

template <int C>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
head_ddim_kernel(const float* __restrict__ X, LnParams post, LnParams head_ln, const float* __restrict__ wh,
                 const float* __restrict__ bh, DdimStep s, float* __restrict__ y, const float* __restrict__ noise,
                 float* __restrict__ out3, float* __restrict__ trace_y, float* __restrict__ trace_x0,
                 int trace_stride, int trace_idx, int64_t T) {
  const int lane = threadIdx.x & 31;
  const int64_t t = static_cast<int64_t>(blockIdx.x) * kWarpsPerCta + (threadIdx.x >> 5);
  if (t >= T) return;
  float x[C / 32], z[C / 32], h[C / 32], w[C / 32];
  load_row(X + t * C, lane, x);
  layernorm_row(x, post.gamma, post.beta, 1e-6f, lane, z);
  layernorm_row(z, head_ln.gamma, head_ln.beta, 1e-5f, lane, h);
  float o[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    load_row_ldg(wh + k * C, lane, w);
    float d = 0.f;
#pragma unroll
    for (int i = 0; i < C / 32; ++i) d = fmaf(h[i], w[i], d);
    o[k] = warp_sum(d) + __ldg(bh + k);
  }
  if (lane < 3) {
    float x0 = lane == 0 ? o[0] : (lane == 1 ? o[1] : o[2]);
    const int64_t e = t * 3 + lane;
    if (out3) {                     // forward_denoise: raw head output (MODEL:255-257)
      out3[e] = x0;
      return;
    }
    if (s.clip) x0 = fminf(fmaxf(x0, -1.0f), 1.0f);          // DIFF:252,256
    float yn;
    if (s.last) {
      yn = x0;                                               // DIFF:283-285
    } else {
      // literal DIFF:295-297, one rounding per torch op (no FMA contraction)
      const float t1 = __fmul_rn(x0, s.sqrt_alpha_next);
      const float t2 = __fdiv_rn(__fsub_rn(y[e], __fmul_rn(s.alpha, x0)), s.sqrt_one_minus);
      yn = __fadd_rn(t1, __fmul_rn(s.c, t2));
      if (noise) yn = __fadd_rn(yn, __fmul_rn(s.sigma, noise[e]));
    }
    y[e] = yn;
    if (trace_y) trace_y[e * trace_stride + trace_idx] = yn;
    if (trace_x0) trace_x0[e * trace_stride + trace_idx] = x0;
  }
}

// head_ddim on two rows per warp (the two LayerNorms' parameters and the three head weight rows loaded once for both)
__device__ __forceinline__ void head_finish(float o0, float o1, float o2, int lane, int64_t t, const DdimStep& s,
                                            float* __restrict__ y, const float* __restrict__ noise, float* __restrict__ out3,
                                            float* __restrict__ trace_y, float* __restrict__ trace_x0, int trace_stride,
                                            int trace_idx) {
  if (lane < 3) {
    float x0 = lane == 0 ? o0 : (lane == 1 ? o1 : o2);
    const int64_t e = t * 3 + lane;
    if (out3) {                     // forward_denoise: raw head output (MODEL:255-257)
      out3[e] = x0;
      return;
    }
    if (s.clip) x0 = fminf(fmaxf(x0, -1.0f), 1.0f);          // DIFF:252,256
    float yn;
    if (s.last) {
      yn = x0;                                               // DIFF:283-285
    } else {
      // literal DIFF:295-297, one rounding per torch op (no FMA contraction)
      const float t1 = __fmul_rn(x0, s.sqrt_alpha_next);
      const float t2 = __fdiv_rn(__fsub_rn(y[e], __fmul_rn(s.alpha, x0)), s.sqrt_one_minus);
      yn = __fadd_rn(t1, __fmul_rn(s.c, t2));
      if (noise) yn = __fadd_rn(yn, __fmul_rn(s.sigma, noise[e]));
    }
    y[e] = yn;
    if (trace_y) trace_y[e * trace_stride + trace_idx] = yn;
    if (trace_x0) trace_x0[e * trace_stride + trace_idx] = x0;
  }
}

template <int C>
__global__ void __launch_bounds__(kWarpsPerCta * 32, D3D_ROWS2_MIN_CTAS)
head_ddim2_kernel(const float* __restrict__ X, LnParams post, LnParams head_ln, const float* __restrict__ wh,
                  const float* __restrict__ bh, DdimStep s, float* __restrict__ y, const float* __restrict__ noise,
                  float* __restrict__ out3, float* __restrict__ trace_y, float* __restrict__ trace_x0,
                  int trace_stride, int trace_idx, int64_t T) {
  const int lane = threadIdx.x & 31;
  const int64_t t = (static_cast<int64_t>(blockIdx.x) * kWarpsPerCta + (threadIdx.x >> 5)) * 2;
  if (t >= T) return;
  const bool two = t + 1 < T;
  float x0[C / 32], x1[C / 32], z0[C / 32], z1[C / 32], w[C / 32];
  load_row(X + t * C, lane, x0);
  load_row(X + (two ? t + 1 : t) * C, lane, x1);
  layernorm_2rows(x0, x1, post.gamma, post.beta, nullptr, 1e-6f, lane, z0, z1);
  layernorm_2rows(z0, z1, head_ln.gamma, head_ln.beta, nullptr, 1e-5f, lane, x0, x1);
  float o0[3], o1[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    load_row_ldg(wh + k * C, lane, w);
    float d0 = 0.f, d1 = 0.f;
#pragma unroll
    for (int i = 0; i < C / 32; ++i) { d0 = fmaf(x0[i], w[i], d0); d1 = fmaf(x1[i], w[i], d1); }
    const float bk = __ldg(bh + k);
    o0[k] = warp_sum(d0) + bk;
    o1[k] = warp_sum(d1) + bk;
  }
  head_finish(o0[0], o0[1], o0[2], lane, t, s, y, noise, out3, trace_y, trace_x0, trace_stride, trace_idx);
  if (two) head_finish(o1[0], o1[1], o1[2], lane, t + 1, s, y, noise, out3, trace_y, trace_x0, trace_stride, trace_idx);
}

__global__ void tta_merge_kernel(const float* __restrict__ y, const float* __restrict__ yf,
                                 const int32_t* __restrict__ perm, float scale, float* __restrict__ out,
                                 int64_t n_elems, int J) {
  const int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e >= n_elems) return;
  const int k = static_cast<int>(e % 3);
  const int64_t fj = e / 3;
  const int j = static_cast<int>(fj % J);
  const int64_t f = fj / J;
  float v = yf[(f * J + perm[j]) * 3 + k];
  if (k == 0) v = -v;
  out[e] = __fmul_rn(__fdiv_rn(__fadd_rn(y[e], v), 2.0f), scale);     // RUN:587-588
}

__global__ void mpjpe_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                             const uint8_t* __restrict__ mask, int64_t n_joints_total, int J,
                             double* __restrict__ acc) {
  double s = 0.0, c = 0.0;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_joints_total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    if (mask && !mask[i / J]) continue;
    const float dx = pred[i * 3] - gt[i * 3], dy = pred[i * 3 + 1] - gt[i * 3 + 1], dz = pred[i * 3 + 2] - gt[i * 3 + 2];
    s += static_cast<double>(sqrtf(dx * dx + dy * dy + dz * dz));
    c += 1.0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    c += __shfl_xor_sync(0xffffffffu, c, o);
  }
  __shared__ double ss[32], cs[32];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { ss[w] = s; cs[w] = c; }
  __syncthreads();
  if (w == 0) {
    s = l < (blockDim.x >> 5) ? ss[l] : 0.0;
    c = l < (blockDim.x >> 5) ? cs[l] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s += __shfl_xor_sync(0xffffffffu, s, o);
      c += __shfl_xor_sync(0xffffffffu, c, o);
    }
    if (l == 0) { atomicAdd(acc, s); atomicAdd(acc + 1, c); }
  }
}

// fp32 [rows, K] -> operand arrays.  is_weight selects the weight-side e5m2 scales of FMT_F8C.
__global__ void split_kernel(const float* __restrict__ in, __half* __restrict__ hi, __half* __restrict__ second,
                             int64_t n, int K, int fmt, int is_weight, float* __restrict__ absmax) {
  float amax = 0.f;
  bool bad = false;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float v = in[i];
    if (isfinite(v)) amax = fmaxf(amax, fabsf(v)); else bad = true;
    const __half h = __float2half_rn(v);
    const float l = v - __half2float(h);
    hi[i] = h;
    if (!second) continue;
    if (fmt == FMT_SPLIT16) {
      second[i] = __float2half_rn(l);
    } else {
      const int64_t row = i / K;
      const int col = static_cast<int>(i - row * K);
      uint8_t* c8 = reinterpret_cast<uint8_t*>(second) + row * 2 * K;
      const float first = is_weight ? l * kWgtLoScale : v * kActHiScale;
      const float secnd = is_weight ? v * kWgtHiScale : l * kActLoScale;
      c8[col] = static_cast<uint8_t>(op_e5m2x2(first, 0.f) & 0xff);
      c8[K + col] = static_cast<uint8_t>(op_e5m2x2(secnd, 0.f) & 0xff);
    }
  }
  if (absmax) {       // non-negative floats order like their bit patterns
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned int*>(absmax), __float_as_uint(amax));
    if (bad) absmax[1] = 1.0f;
  }
}
// FMT_F4C split: one thread per 32-element block (row, kb) of the [rows, K] input: hi, both nibble parts and both scale
// bytes.  Activations: P = q4(x), Q = q4(x - hi); weights: P = q4(w - hi), Q = q4(w)  (operand.cuh).
__global__ void split_f4c_kernel(const float* __restrict__ in, __half* __restrict__ hi, uint8_t* __restrict__ c4,
                                 uint8_t* __restrict__ sf, int64_t rows, int K, int is_weight, float* __restrict__ absmax) {
  const int bpr = K / 32;                       // blocks per row and part
  const int64_t n_blocks = rows * bpr;
  float amax_all = 0.f;
  bool bad = false;
  for (int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; b < n_blocks;
       b += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t row = b / bpr;
    const int kb = static_cast<int>(b - row * bpr);
    const float* src = in + row * K + kb * 32;
    float x[32], l[32];
    float ax = 0.f, al = 0.f;
#pragma unroll
    for (int e = 0; e < 32; e += 4) {
      const float4 t = *reinterpret_cast<const float4*>(src + e);
      x[e] = t.x; x[e + 1] = t.y; x[e + 2] = t.z; x[e + 3] = t.w;
    }
    uint32_t hw[16];
#pragma unroll
    for (int e = 0; e < 32; e += 2) {
      const __half h0 = __float2half_rn(x[e]), h1 = __float2half_rn(x[e + 1]);
      hw[e >> 1] = op_pack_h2(h0, h1);
      l[e] = x[e] - __half2float(h0);
      l[e + 1] = x[e + 1] - __half2float(h1);
    }
#pragma unroll
    for (int e = 0; e < 32; ++e) {
      if (!isfinite(x[e])) bad = true;
      ax = fmaxf(ax, fabsf(x[e]));
      al = fmaxf(al, fabsf(l[e]));
    }
    amax_all = fmaxf(amax_all, ax);
    uint4* hdst = reinterpret_cast<uint4*>(hi + row * K + kb * 32);
#pragma unroll
    for (int q = 0; q < 4; ++q) hdst[q] = make_uint4(hw[4 * q], hw[4 * q + 1], hw[4 * q + 2], hw[4 * q + 3]);
    const float* pv = is_weight ? l : x;       // part P
    const float* qv = is_weight ? x : l;       // part Q
    const uint32_t bp = op_ue8m0_of(is_weight ? al : ax), bq = op_ue8m0_of(is_weight ? ax : al);
    const float ip = op_ue8m0_inv(bp), iq = op_ue8m0_inv(bq);
    uint8_t* crow = c4 + row * K;
    *reinterpret_cast<uint4*>(crow + kb * 16) =
        make_uint4(op_e2m1x8(pv, ip), op_e2m1x8(pv + 8, ip), op_e2m1x8(pv + 16, ip), op_e2m1x8(pv + 24, ip));
    *reinterpret_cast<uint4*>(crow + (K >> 1) + kb * 16) =
        make_uint4(op_e2m1x8(qv, iq), op_e2m1x8(qv + 8, iq), op_e2m1x8(qv + 16, iq), op_e2m1x8(qv + 24, iq));
    sf[op_sf_offset(row, kb, K / 64)] = static_cast<uint8_t>(bp);
    sf[op_sf_offset(row, bpr + kb, K / 64)] = static_cast<uint8_t>(bq);
  }
  if (absmax) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) amax_all = fmaxf(amax_all, __shfl_xor_sync(0xffffffffu, amax_all, o));
    if ((threadIdx.x & 31) == 0 && isfinite(amax_all)) atomicMax(reinterpret_cast<unsigned int*>(absmax), __float_as_uint(amax_all));
    if (bad) absmax[1] = 1.0f;
  }
}
// FMT_F4C activation operand -> fp32: hi + q4(Q) * scale
__global__ void merge_f4c_kernel(const __half* __restrict__ hi, const uint8_t* __restrict__ c4, const uint8_t* __restrict__ sf,
                                 float* __restrict__ out, int64_t n, int K) {
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t row = i / K;
    const int col = static_cast<int>(i - row * K);
    const uint32_t byte = c4[row * K + (K >> 1) + (col >> 1)];
    const float q = op_e2m1_to_float((col & 1) ? (byte >> 4) : (byte & 15u));
    const float sc = op_ue8m0_val(sf[op_sf_offset(row, K / 32 + col / 32, K / 64)]);
    out[i] = __half2float(hi[i]) + q * sc;
  }
}

// scale-factor atoms -> row-major [rows][K / 16] bytes (test read-back of a FMT_F4C operand)
__global__ void sf_rows_kernel(const uint8_t* __restrict__ sf, uint8_t* __restrict__ out, int64_t n, int K) {
  const int per_row = K / 16;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t row = i / per_row;
    out[i] = sf[op_sf_offset(row, static_cast<int>(i - row * per_row), K / 64)];
  }
}

// activation operand -> fp32 (hi + lo); for FMT_F8C the lo term comes back from its e5m2 image
__global__ void merge_kernel(const __half* __restrict__ hi, const __half* __restrict__ second, float* __restrict__ out,
                             int64_t n, int K, int fmt) {
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float lo;
    if (fmt == FMT_SPLIT16) {
      lo = __half2float(second[i]);
    } else {
      const int64_t row = i / K;
      const int col = static_cast<int>(i - row * K);
      lo = op_e5m2_to_float(reinterpret_cast<const uint8_t*>(second)[row * 2 * K + K + col]) * (1.0f / kActLoScale);
    }
    out[i] = __half2float(hi[i]) + lo;
  }
}

// D3D_LN_ROWS = 1: the one-row-per-warp forms of ln_split / postnorm_add_ln (A/B; read when the launch sequence is built)
inline int rows_per_warp() {
  const char* v = getenv("D3D_LN_ROWS");
  return (v && *v == '1') ? 1 : 2;
}
inline unsigned row_grid(int64_t T) { return static_cast<unsigned>((T + kWarpsPerCta - 1) / kWarpsPerCta); }
inline unsigned flat_grid(int64_t n) {
  int64_t g = (n + 255) / 256;
  return static_cast<unsigned>(g > 148 * 32 ? 148 * 32 : (g < 1 ? 1 : g));
}

}  // namespace

cudaError_t launch_split(const float* in, __half* hi, __half* second, uint8_t* sf, int64_t rows, int K, int fmt,
                         int is_weight, cudaStream_t st, float* absmax) {
  const int64_t n = rows * K;
  if (n <= 0) return cudaSuccess;
  if (fmt == FMT_F4C) {
    if (K % 64 != 0 || !sf || !second) return cudaErrorInvalidValue;
    split_f4c_kernel<<<flat_grid(n / 32), 128, 0, st>>>(in, hi, reinterpret_cast<uint8_t*>(second), sf, rows, K, is_weight,
                                                       absmax);
  } else {
    split_kernel<<<flat_grid(n), 256, 0, st>>>(in, hi, second, n, K, fmt, is_weight, absmax);
  }
  return cudaGetLastError();
}
cudaError_t launch_merge(const __half* hi, const __half* second, const uint8_t* sf, float* out, int64_t rows, int K,
                         int fmt, cudaStream_t st) {
  const int64_t n = rows * K;
  if (n <= 0) return cudaSuccess;
  if (fmt == FMT_F4C) merge_f4c_kernel<<<flat_grid(n), 256, 0, st>>>(hi, reinterpret_cast<const uint8_t*>(second), sf, out, n, K);
  else merge_kernel<<<flat_grid(n), 256, 0, st>>>(hi, second, out, n, K, fmt);
  return cudaGetLastError();
}
cudaError_t launch_sf_rows(const uint8_t* sf, uint8_t* out, int64_t rows, int K, cudaStream_t st) {
  const int64_t n = rows * (K / 16);
  if (n <= 0) return cudaSuccess;
  sf_rows_kernel<<<flat_grid(n), 256, 0, st>>>(sf, out, n, K);
  return cudaGetLastError();
}
// The (C, FMT) instantiation of a row-wise kernel: every operand format at C = 512, the shipped FMT_F4C at C = 256.
inline bool rowwise_built(int C, int fmt) { return C == 512 || (C == 256 && fmt == FMT_F4C); }
#define D3D_ROWWISE_PICK(KERN)                                                                                          \
  (C == 256 ? KERN<256, FMT_F4C> : fmt == FMT_F4C ? KERN<512, FMT_F4C> : fmt == FMT_F8C ? KERN<512, FMT_F8C> \
                                                                                 : KERN<512, FMT_SPLIT16>)

cudaError_t launch_lift_ln(int C, const float* x2d, const float* y, const float* x5, const float* wf_t, const float* bf,
                           const float* spos, const float* tvec, int64_t tvec_stride, LnParams ln1, float* X,
                           __half* a_hi, __half* a_lo, uint8_t* a_sf, int fmt, int64_t T, int J, int tokens_per_clip,
                           cudaStream_t st) {
  if (T <= 0) return cudaSuccess;
  if (T > 0x7fffffffLL || !rowwise_built(C, fmt)) return cudaErrorInvalidValue;
  if ((!tvec || tvec_stride == 0) && rows_per_warp() == 2) {
    auto k2 = D3D_ROWWISE_PICK(lift_ln2_kernel);
    k2<<<row_grid((T + 1) / 2), kWarpsPerCta * 32, 0, st>>>(x2d, y, x5, wf_t, bf, spos, tvec, ln1, X, a_hi, a_lo, a_sf, T, J);
    return cudaGetLastError();
  }
  auto kern = D3D_ROWWISE_PICK(lift_ln_kernel);
  kern<<<row_grid(T), kWarpsPerCta * 32, 0, st>>>(x2d, y, x5, wf_t, bf, spos, tvec, tvec_stride, ln1, X, a_hi, a_lo, a_sf, T,
                                                 J, tokens_per_clip);
  return cudaGetLastError();
}
cudaError_t launch_postnorm_add_ln(int C, float* X, LnParams post, const float* tpos, const float* tvec,
                                   int64_t tvec_stride, LnParams ln1, __half* a_hi, __half* a_lo, uint8_t* a_sf, int fmt,
                                   int64_t T, int J, int F, cudaStream_t st) {
  if (T <= 0) return cudaSuccess;
  if (T > 0x7fffffffLL || !rowwise_built(C, fmt)) return cudaErrorInvalidValue;
  if (!tpos && (!tvec || tvec_stride == 0) && rows_per_warp() == 2) {       // eval: no per-row additive term
    auto k2 = D3D_ROWWISE_PICK(postnorm_add_ln2_kernel);
    k2<<<row_grid((T + 1) / 2), kWarpsPerCta * 32, 0, st>>>(X, post, tvec, ln1, a_hi, a_lo, a_sf, T);
    return cudaGetLastError();
  }
  auto kern = D3D_ROWWISE_PICK(postnorm_add_ln_kernel);
  kern<<<row_grid(T), kWarpsPerCta * 32, 0, st>>>(X, post, tpos, tvec, tvec_stride, ln1, a_hi, a_lo, a_sf, T, J, F);
  return cudaGetLastError();
}
cudaError_t launch_ln_split(int C, const float* X, LnParams ln, float eps, __half* a_hi, __half* a_lo, uint8_t* a_sf,
                            int fmt, int64_t T, cudaStream_t st) {
  if (T <= 0) return cudaSuccess;
  if (!rowwise_built(C, fmt)) return cudaErrorInvalidValue;
  if (rows_per_warp() == 2) {
    auto k2 = D3D_ROWWISE_PICK(ln_split2_kernel);
    k2<<<row_grid((T + 1) / 2), kWarpsPerCta * 32, 0, st>>>(X, ln, eps, a_hi, a_lo, a_sf, T);
    return cudaGetLastError();
  }
  auto kern = D3D_ROWWISE_PICK(ln_split_kernel);
  kern<<<row_grid(T), kWarpsPerCta * 32, 0, st>>>(X, ln, eps, a_hi, a_lo, a_sf, T);
  return cudaGetLastError();
}
#undef D3D_ROWWISE_PICK
cudaError_t launch_ln_f32(int C, const float* x, LnParams ln, float eps, float* out, int64_t T, cudaStream_t st) {
  if (T <= 0) return cudaSuccess;
  if (!width_supported(C)) return cudaErrorInvalidValue;
  auto kern = C == 256 ? ln_f32_kernel<256> : ln_f32_kernel<512>;
  kern<<<row_grid(T), kWarpsPerCta * 32, 0, st>>>(x, ln, eps, out, T);
  return cudaGetLastError();
}
cudaError_t launch_head_ddim(int C, const float* X, LnParams post, LnParams head_ln, const float* wh, const float* bh,
                             DdimStep s, float* y, const float* noise, float* out3, float* trace_y, float* trace_x0,
                             int trace_stride, int trace_idx, int64_t T, cudaStream_t st) {
  if (T <= 0) return cudaSuccess;
  if (!width_supported(C)) return cudaErrorInvalidValue;
  if (rows_per_warp() == 2) {
    auto kern = C == 256 ? head_ddim2_kernel<256> : head_ddim2_kernel<512>;
    kern<<<row_grid((T + 1) / 2), kWarpsPerCta * 32, 0, st>>>(X, post, head_ln, wh, bh, s, y, noise, out3, trace_y, trace_x0,
                                                             trace_stride, trace_idx, T);
  } else {
    auto kern = C == 256 ? head_ddim_kernel<256> : head_ddim_kernel<512>;
    kern<<<row_grid(T), kWarpsPerCta * 32, 0, st>>>(X, post, head_ln, wh, bh, s, y, noise, out3, trace_y, trace_x0,
                                                   trace_stride, trace_idx, T);
  }
  return cudaGetLastError();
}
cudaError_t launch_tta_merge(const float* y, const float* yf, const int32_t* perm, float scale, float* out,
                             int64_t n_frames, int J, cudaStream_t st) {
  const int64_t n = n_frames * J * 3;
  if (n <= 0) return cudaSuccess;
  tta_merge_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(y, yf, perm, scale, out, n, J);
  return cudaGetLastError();
}
cudaError_t launch_mpjpe(const float* pred, const float* gt, const uint8_t* mask, int64_t n_frames, int J,
                         double* acc, cudaStream_t st) {
  const int64_t n = n_frames * J;
  if (n <= 0) return cudaSuccess;
  mpjpe_kernel<<<flat_grid(n), 256, 0, st>>>(pred, gt, mask, n, J, acc);
  return cudaGetLastError();
}

}  // namespace d3d
