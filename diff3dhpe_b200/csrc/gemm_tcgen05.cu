// G-gemm: the qkv / proj / fc1 / fc2 linears of MixSTE (MODEL:75, 84, 51-54) as a persistent,
// warp-specialised tcgen05 GEMM for sm_100a.
//
//   out[M,N] = epilogue( A[M,K] . W[N,K]^T + bias[N] )
//
//   * operands are fp16 "split halves": x = hi + lo with hi = fp16(x), lo = fp16(x - hi).  The default
//     3-pass mode issues   D += A_hi.B_hi ; D += A_hi.B_lo ; D += A_lo.B_hi   per k-step, accumulating in
//     fp32 in TMEM, which restores ~22 mantissa bits (SURVEY.md 7.3-1: single-pass bf16/fp16 misses the
//     parity bar).  The 1-pass mode issues only A_hi.B_hi.  PASSES == 2 is the FMT_F8C mode of operand.cuh: the
//     fp16 main product followed by ONE kind::f8f6f4 (e5m2) product over K' = 2K that carries both correction
//     terms -- 2 tensor-pipe units instead of 3; the second tensor maps then describe the uint8 c8 arrays and
//     the ring holds 2 * K/64 uniform stages per tile (fp16 stages first, then fp8 stages).  PASSES == 4 is FMT_F4C:
//     the correction product in block-scaled e2m1 (kind::mxf4.block_scale, 4x the fp16 rate; 1.5 units): K/64 fp16
//     stages, then K/128 stages of 256 e2m1 each that also carry the stage's ue8m0 scale-factor atoms (3 KB), which the
//     MMA thread copies into TMEM with tcgen05.cp right before the stage's four MMAs.  The scale columns live in the
//     first 32 columns of the OTHER accumulator, which the previous tile's epilogue has drained by then (see sf_free).
//   * TMA (cp.async.bulk.tensor, SWIZZLE_128B) stages {128 rows x 64} fp16 boxes; a ring of mbarrier-guarded
//     stages feeds one MMA-issuing thread.
//   * CG = 2 (default): a CTA PAIR (thread-block cluster of 2, tcgen05.mma.cta_group::2) owns a 256 x 256
//     output tile.  Each CTA stages its own 128 rows of A and HALF of the 256 weight rows, so the L2 -> SM
//     operand traffic per MAC is 2/3 of the single-CTA 128 x 256 tile.  ncu on the single-CTA kernel
//     (profiles/r01a) showed lts__throughput at the ~6300 B/clk L2 cap with the tensor pipe only 52 % busy:
//     operand bytes per MAC, not MMA issue, bound this GEMM.  The leader CTA (cluster rank 0) issues the MMAs
//     for both; its tcgen05.commit multicasts "stage free" / "accumulator ready" to both CTAs' mbarriers.
//     CG = 1 keeps the single-CTA 128 x BN kernel (validation / small problems).
//   * accumulators are double-buffered in TMEM (2 x 256 fp32 columns) so the epilogue of tile i overlaps the
//     mainloop of tile i+1.  Eight epilogue warps per CTA read TMEM with tcgen05.ld (32 lanes x 32 columns);
//     the residual rows of chunk c+1 are prefetched while chunk c is in flight (the un-prefetched version was
//     latency-bound: 26 % tensor-pipe on the proj GEMM).
//   * epilogues (kernels.cuh GemmEpi): fp32 (+ residual) through a swizzled transpose buffer; the SHIPPED in-place residual
//     update of proj / fc2 as a TMA reduction (EPI_F32_RED: the L2 adds, X never enters the SM -- the L2 -> SM operand
//     feed is what bounds all four GEMMs, DESIGN.md 4.1); q | k | v_hi | v_lo fp16 pack; GELU -> block-scaled operand (1-MUFU
//     GELU, bias from shared memory, per-lane store addressing); the deferred-LayerNorm pair EPI_F32_EMIT / EPI_GELU_DLN
//     (measured, off by default).
//
// Warp roles (384 threads): 0 = TMA producer, 1 = MMA issuer (leader CTA), 2 = TMEM allocator, 3 = idle,
// 4..11 = epilogue (EW = 16: 640 threads, epilogue warps 4..19, setmaxnreg 32 / 112).
#include <cstdlib>
#include "kernels.cuh"
#include "operand.cuh"
#include "ptx.cuh"

namespace d3d {

namespace {

constexpr int BM = 128;                      // rows per CTA
constexpr int BK = 64;                       // 64 fp16 = 128 B = one swizzle row
#ifndef D3D_GEMM_PRODUCER_REGS
#define D3D_GEMM_PRODUCER_REGS 32          // 32 / 112 (round 2): no spills left in the 16-warp fp32 / GELU epilogues
#define D3D_GEMM_EPILOGUE_REGS 112
#endif
constexpr int kProducerRegs = D3D_GEMM_PRODUCER_REGS;   // setmaxnreg targets of the EW = 16 kernels (640 threads launch with 96 each)
constexpr int kEpilogueRegs = D3D_GEMM_EPILOGUE_REGS;
// setmaxnreg.inc draws from the registers the SAME CTA released with setmaxnreg.dec (not from the SM's unallocated
// remainder): the four epilogue warpgroups may not ask for more than the producer warpgroup gave back, or they block
// forever (first attempt: 40 / 112 -> deadlock on the GPU)
static_assert(4 * 128 * (kEpilogueRegs - 96) <= 128 * (96 - kProducerRegs), "setmaxnreg pool overdrawn");
constexpr int kTileBytesA = BM * BK * 2;     // 16 KiB
#ifndef D3D_GEMM_SMEM_BUDGET_KB
#define D3D_GEMM_SMEM_BUDGET_KB 200
#endif
constexpr int kSmemBudget = D3D_GEMM_SMEM_BUDGET_KB * 1024;   // ring + epilogue staging (A/B builds: fewer ring stages)

// EW = epilogue warps per CTA: 8 (two warps per TMEM lane quadrant, 128 columns each) or 16 (four per quadrant, 64
// columns each).  The bias+GELU+split epilogue of fc1 costs ~25 instructions per output element; with 8 warps it, not
// the MMA or L2, bounded that GEMM (11.9 us per 256 x 256 tile against 8.6 us for the qkv GEMM at the same K).
template <int CG, int BN, int PASSES, int EW = 8>
struct Cfg {
  static constexpr int kBRows = BN / CG;                  // weight rows staged by one CTA
  static constexpr int kTileBytesB = kBRows * BK * 2;
  static constexpr int kThreads = 128 + 32 * EW;
  // FMT_F4C: every ring slot has room for the scale-factor atoms of an e2m1 stage behind the A / B tiles:
  // A: 128 rows x 8 k-blocks = 1 KB, B: 256 rows (BOTH halves: each CTA's MMA scales all 256 columns) x 8 = 2 KB
  static constexpr int kSfBytes = PASSES == 4 ? 3072 : 0;
  static constexpr int kStageBytes = (PASSES == 3 ? 2 : 1) * (kTileBytesA + kTileBytesB) + kSfBytes;
  static constexpr int kStagingBytes = EW * 4096;   // one 32-row x 128-byte transpose buffer per epilogue warp
  static constexpr int kRing = ((PASSES == 2 || PASSES == 4) ? kSmemBudget : 200 * 1024) + 8 * 4096 - kStagingBytes;   // + 8 KB vectors (F4C)
  static constexpr int kStages = (kRing / kStageBytes) > 8 ? 8 : (kRing / kStageBytes);
  static constexpr int kTmemCols = 2 * BN;   // 256 or 512 (power of two)
  // FMT_F4C operand-producing epilogues (GELU / deferred LayerNorm) read bias (and the folded weight's column sums) from
  // shared memory, just in time, instead of holding 32 prefetched registers per lane across the accumulator wait
  static constexpr int kVecBytes = PASSES == 4 ? 2 * 1024 * 4 : 0;
  static constexpr int kSmemBytes = kStages * kStageBytes + kStagingBytes + 1024 /*align*/ + 256 /*barriers*/ + kVecBytes;
  static_assert(kStages >= 2, "need at least a double buffer");
  static_assert(CG == 1 || BN == 256, "the CTA-pair kernel uses 256 x 256 tiles");
  static_assert(EW == 8 || (EW == 16 && BN == 256), "16 epilogue warps split a 256-column tile four ways");
  static_assert(PASSES != 4 || (CG == 2 && BN == 256), "the F4C kernel is the CTA-pair 256 x 256 kernel");
  static_assert(kStageBytes % 1024 == 0, "SWIZZLE_128B tiles need 1024-byte aligned stages");
};

struct Barriers {
  uint64_t full[8];
  uint64_t empty[8];
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint64_t sf_free[2];     // F4C: the first 32 columns of accumulator a have been read by the epilogue (both CTAs)
  uint32_t tmem_base;
};

#ifndef D3D_GEMM_RES_DEPTH
#define D3D_GEMM_RES_DEPTH 2     // residual chunks prefetched per epilogue warp (A/B builds: 1 = the round-1 epilogue)
#endif

// D3D_EPI_PACKED = 0 compiles the scalar epilogue math (the A/B baseline of profiles/r01z_bench_scalar_epilogue.json)
#ifndef D3D_EPI_PACKED
#define D3D_EPI_PACKED 1
#endif

// Exact-erf GELU (MODEL:52, nn.GELU()) without the branchy library erff: the epilogue is instruction-issue bound
// (32 768 activations per 128 x 256 tile), so the form below is branch- and call-free, 2 MUFU + ~14 FP32 ops:
//   gelu(v) = max(v, 0) - |v|/2 * erfc(|v| / sqrt 2),   erfc(z) = t (a1 + t (a2 + t (a3 + t (a4 + t a5)))) exp(-z^2),
//   t = 1 / (1 + p z)   (Abramowitz-Stegun 7.1.26, |error| <= 1.5e-7 on erfc; using erfc for BOTH signs avoids the
//   1 + erf cancellation in the negative tail).  Absolute error on gelu <= |v| * 1e-7.
#if !D3D_EPI_PACKED
__device__ __forceinline__ float gelu_erf(float v) {
  const float z = fabsf(v) * 0.70710678118654752440f;
  float t, e;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.0f)));      // MUFU, rel. error 2^-23
  float poly = fmaf(t, 1.061405429f, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.4426950408889634f * z * z));   // MUFU, rel. error 2^-22
  return fmaxf(v, 0.0f) - (0.70710678118654752440f * z) * (poly * t * e);
}
#endif

// The same function on a PACKED pair (FFMA2 / FMUL2: two IEEE-rn operations per fma-pipe slot; D3D_GELU_POLY5 = 0 builds
// this form, the round-1 epilogue).  The scalar form costs
// 16 fma-pipe instructions per activation incl. bias and operand split; a 3-register FFMA issues every other cycle per
// scheduler, so 32 768 activations per CTA tile kept the fma pipe busy for ~8 200 cycles -- longer than the tile's
// mainloop.  Constants are folded so that no scaling multiply is left: with a = |v|,
//   t = 1 / (1 + (p / sqrt 2) a),  e = exp2(-(log2 e / 2) a^2),  q(t) = -(a1 + t (a2 + ...)) / 2   (exact scaling),
//   gelu(v) = max(v, 0) + a (q(t) t e).
// D3D_GELU_POLY5 = 1 (default): ONE MUFU per activation.  With a = |v| and Q(a) = erfc(a / sqrt 2) / 2 (the normal tail),
//   gelu(v) = v / 2 + a (1/2 - Q(a)),   Q(a) = exp2(p(a)),  p = degree-5 minimax fit of log2 Q weighted by the sensitivity
//   a Q(a) of the result (tools/fit_gelu_tail.py): |error| <= 4.8e-7 absolute for every v (the A-S form: <= |v| 1e-7;
//   both far below the 6e-5 relative precision of the operand format the result is written in).  p's leading coefficient
//   is negative, so Q underflows to 0 for large a and gelu(v) -> max(v, 0) without a clamp.  5 + 3 packed fma-pipe
//   instructions and 1 MUFU per activation instead of 10 + 2 (+ the scalar max): the fc1 epilogue is issue-bound.
#ifndef D3D_GELU_POLY5
#define D3D_GELU_POLY5 1
#endif
#if D3D_EPI_PACKED && D3D_GELU_POLY5
__device__ __forceinline__ ptx::f32x2 gelu_erf2(ptx::f32x2 v) {
  float v0, v1, g0, g1, e0, e1;
  ptx::unpack2(v, v0, v1);
  const ptx::f32x2 a = ptx::pack2(fabsf(v0), fabsf(v1));
  ptx::f32x2 q = ptx::fma2(a, ptx::splat2(-4.732940288e-04f), ptx::splat2(7.084461395e-03f));
  q = ptx::fma2(q, a, ptx::splat2(-5.182716995e-02f));
  q = ptx::fma2(q, a, ptx::splat2(-4.599926472e-01f));
  q = ptx::fma2(q, a, ptx::splat2(-1.150787711e+00f));
  q = ptx::fma2(q, a, ptx::splat2(-1.000037670e+00f));
  ptx::unpack2(q, g0, g1);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(g0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(g1));
  const ptx::f32x2 h = ptx::sub2(ptx::splat2(0.5f), ptx::pack2(e0, e1));
  return ptx::fma2(a, h, ptx::mul2(v, ptx::splat2(0.5f)));
}
#elif D3D_EPI_PACKED
__device__ __forceinline__ ptx::f32x2 gelu_erf2(ptx::f32x2 v) {
  float v0, v1;
  ptx::unpack2(v, v0, v1);
  const ptx::f32x2 a = ptx::pack2(fabsf(v0), fabsf(v1));
  float d0, d1, t0, t1, g0, g1, e0, e1;
  ptx::unpack2(ptx::fma2(a, ptx::splat2(0.3275911f * 0.70710678118654752440f), ptx::splat2(1.0f)), d0, d1);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t0) : "f"(d0));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t1) : "f"(d1));
  const ptx::f32x2 t = ptx::pack2(t0, t1);
  ptx::f32x2 q = ptx::fma2(t, ptx::splat2(-0.5f * 1.061405429f), ptx::splat2(0.5f * 1.453152027f));
  q = ptx::fma2(q, t, ptx::splat2(-0.5f * 1.421413741f));
  q = ptx::fma2(q, t, ptx::splat2(0.5f * 0.284496736f));
  q = ptx::fma2(q, t, ptx::splat2(-0.5f * 0.254829592f));
  ptx::unpack2(ptx::mul2(ptx::mul2(a, a), ptx::splat2(-0.5f * 1.4426950408889634f)), g0, g1);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(g0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(g1));
  const ptx::f32x2 w = ptx::mul2(ptx::mul2(q, t), ptx::pack2(e0, e1));
  return ptx::fma2(a, w, ptx::pack2(fmaxf(v0, 0.0f), fmaxf(v1, 0.0f)));
}
#endif

// Epilogue transpose buffer: 32 rows x 128 B; the 16-byte granule g of row r lives at r*128 + ((g ^ (r&7)) << 4)
// (the 128-byte swizzle), so "lane = row" accesses and "8 lanes = one row" accesses are both conflict-free.
// The accessors take the buffer's shared-space (32-bit) address: one ld / st.shared with 32-bit address arithmetic per
// access (through a generic pointer every access cost a 64-bit add and a generic-space instruction).
__device__ __forceinline__ uint32_t stg_at(uint32_t stg, int r, int g) { return stg + r * 128 + ((g ^ (r & 7)) << 4); }
__device__ __forceinline__ void stg_st(uint32_t stg, int r, int g, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg_at(stg, r, g)), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}
__device__ __forceinline__ uint4 stg_ld(uint32_t stg, int r, int g) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(stg_at(stg, r, g))
               : "memory");
  return v;
}
// read-only per-column vectors in shared memory (written once before the role split): schedulable like any load
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}

__device__ __forceinline__ uint32_t pack_h2(__half a, __half b) {
  return static_cast<uint32_t>(__half_as_ushort(a)) | (static_cast<uint32_t>(__half_as_ushort(b)) << 16);
}

// Coalesced stores of one FMT_F4C staging buffer (32 rows x 128 B: granules 0..3 = 32 hi halves, 4 = 32 P nibbles,
// 5 = 32 Q nibbles; 8 lanes = one row).  Which array a lane writes depends only on its granule, so base pointer and row
// pitch are per-lane constants of the whole kernel: a store costs one 64-bit add, no divergent address code (the first
// version re-derived the three-way address per store: a quarter of the fc1 epilogue's instructions).
struct F4cStore {
  uint8_t* base;     // hi: out_hi + 16 gsub bytes;  P: c4;  Q: c4 + N / 2
  size_t pitch;      // bytes per row: 2 N (hi) or N (c4)
  int col_shift;     // byte offset of column c inside the row: c << 1 (hi) or c >> 1 (nibbles)
  bool on;           // granules 6, 7 carry nothing
};
__device__ __forceinline__ F4cStore f4c_store_init(__half* out_hi, uint8_t* c4, int N, int gsub) {
  F4cStore st;
  const bool hi = gsub < 4;
  st.base = hi ? reinterpret_cast<uint8_t*>(out_hi) + gsub * 16 : c4 + (gsub == 5 ? (N >> 1) : 0);
  st.pitch = hi ? static_cast<size_t>(2 * N) : static_cast<size_t>(N);
  st.col_shift = hi ? 1 : -1;
  st.on = gsub < 6;
  return st;
}
__device__ __forceinline__ void f4c_store_chunk(const F4cStore& st, uint32_t stg, int rsub, int gsub, int row_w, int gcol,
                                                int M, bool stream_out) {
  uint4 vals[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) vals[j] = stg_ld(stg, 4 * j + rsub, gsub);
  uint8_t* d = st.base + static_cast<size_t>(row_w + rsub) * st.pitch + (st.col_shift > 0 ? gcol << 1 : gcol >> 1);
  const size_t step = 4 * st.pitch;
  if (M - row_w >= 32) {                           // warp-uniform: whole chunk inside the matrix, no per-store predicate
    if (st.on) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (stream_out) ptx::st_global_cs(d, vals[j]); else *reinterpret_cast<uint4*>(d) = vals[j];
        d += step;
      }
    }
    return;
  }
  const int rows_left = M - row_w - rsub;          // ragged last tile: row 4 j + rsub is stored while 4 j < rows_left
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (st.on && 4 * j < rows_left) {
      if (stream_out) ptx::st_global_cs(d, vals[j]); else *reinterpret_cast<uint4*>(d) = vals[j];
    }
    d += step;
  }
}

// FMT_F4C image of one 32 x 32 chunk of fp32 values (lane = row, r = the bits of its 32 consecutive columns = exactly one
// scale block of each part): hi halves into the staging row (granules 0..3) with the block maxima of x and of x - hi, then
// both e2m1 images (granule 4 = 32 nibbles of P = q4(x), granule 5 = Q = q4(x - hi)), then the coalesced stores.  The two
// ue8m0 scale bytes join the lane's words (byte (gcol / 32) % 4); the caller writes them once per tile.
__device__ __forceinline__ void f4c_emit_chunk(const uint32_t (&r)[32], uint32_t stg, int lane, int row_w, int gcol, int M,
                                               const F4cStore& st, bool stream_out, uint32_t& sfp_w, uint32_t& sfq_w) {
  float ax = 0.f, al = 0.f;
#pragma unroll
  for (int v = 0; v < 4; ++v) {
    uint32_t hw[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float x0 = __uint_as_float(r[8 * v + 2 * e + 0]), x1 = __uint_as_float(r[8 * v + 2 * e + 1]);
      const __half2 h01 = __floats2half2_rn(x0, x1);
      const float2 hf = __half22float2(h01);
      hw[e] = *reinterpret_cast<const uint32_t*>(&h01);
      ax = fmaxf(ax, fmaxf(fabsf(x0), fabsf(x1)));
      al = fmaxf(al, fmaxf(fabsf(x0 - hf.x), fabsf(x1 - hf.y)));
    }
    stg_st(stg, lane, v, make_uint4(hw[0], hw[1], hw[2], hw[3]));
  }
  const uint32_t bp = op_ue8m0_of(ax), bq = op_ue8m0_of(al);
  const ptx::f32x2 ip = ptx::splat2(op_ue8m0_inv(bp)), iq = ptx::splat2(op_ue8m0_inv(bq));
  uint32_t pw[4], qw[4];
#pragma unroll
  for (int w = 0; w < 4; ++w) {
    uint32_t pa = 0, qa = 0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float x0 = __uint_as_float(r[8 * w + 2 * e + 0]), x1 = __uint_as_float(r[8 * w + 2 * e + 1]);
      const float2 hf = __half22float2(__floats2half2_rn(x0, x1));
      float a0, a1, l0, l1;
      ptx::unpack2(ptx::mul2(ptx::pack2(x0, x1), ip), a0, a1);
      ptx::unpack2(ptx::mul2(ptx::sub2(ptx::pack2(x0, x1), ptx::pack2(hf.x, hf.y)), iq), l0, l1);
      pa |= op_e2m1x2(a0, a1) << (8 * e);
      qa |= op_e2m1x2(l0, l1) << (8 * e);
    }
    pw[w] = pa; qw[w] = qa;
  }
  stg_st(stg, lane, 4, make_uint4(pw[0], pw[1], pw[2], pw[3]));
  stg_st(stg, lane, 5, make_uint4(qw[0], qw[1], qw[2], qw[3]));
  sfp_w |= bp << (8 * ((gcol >> 5) & 3));
  sfq_w |= bq << (8 * ((gcol >> 5) & 3));
  __syncwarp();
  f4c_store_chunk(st, stg, lane >> 3, lane & 7, row_w, gcol, M, stream_out);
}

// CS = CTA pairs per cluster (CG == 2 only).  CS == 2: a cluster of 4 CTAs owns two vertically adjacent 256 x 256
// tiles (same weight rows).  Each CTA loads only HALF of its 128-row weight tile and TMA-multicasts it to the CTA
// with the same position in the other pair, so the L2 -> SM weight traffic per MAC halves (48 KB instead of 64 KB
// per k-block and SM): the F8C GEMM runs at the ~6300 B/clk L2 output cap (profiles/r01e_full_gemm_tc.md).
template <int CG, int BN, int PASSES, int EPI, int CS, int EW = 8>
__global__ void __launch_bounds__(128 + 32 * EW, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
               const __grid_constant__ CUtensorMap tm_b_hi, const __grid_constant__ CUtensorMap tm_b_lo,
               const __grid_constant__ CUtensorMap tm_a_sf, const __grid_constant__ CUtensorMap tm_b_sf,
               const __grid_constant__ CUtensorMap tm_out, const GemmParams p) {
  using C = Cfg<CG, BN, PASSES, EW>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* staging = smem + C::kStages * C::kStageBytes;
  Barriers* bars = reinterpret_cast<Barriers*>(staging + C::kStagingBytes);
  float* sm_bias = reinterpret_cast<float*>(staging + C::kStagingBytes + 256);      // [1024] bias, [1024] column sums
  float* sm_colsum = sm_bias + 1024;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  static_assert(CS == 1 || (CG == 2 && PASSES == 2), "pair clusters are implemented for the CTA-pair F8C kernel");
  static_assert(PASSES != 4 || EPI != EPI_F32_LN, "the fused LayerNorm epilogue keeps x in TMEM: no room for scale factors");
  static_assert(PASSES == 4 || (EPI != EPI_F32_EMIT && EPI != EPI_GELU_DLN), "deferred LayerNorm: FMT_F4C kernel only");
  constexpr bool kF32 = EPI == EPI_F32 || EPI == EPI_F32_LN || EPI == EPI_F32_EMIT;          // fp32 output (+ residual)
  static_assert(EPI != EPI_F32_RED || PASSES == 4, "the reduction epilogue is built for the FMT_F4C kernel");
  constexpr bool kGelu4 = (EPI == EPI_GELU_SPLIT || EPI == EPI_GELU_DLN) && PASSES == 4;      // GELU -> FMT_F4C operand
  const uint32_t crank = CG == 2 ? ptx::cluster_ctarank() : 0u;     // rank in the cluster (0 .. 2*CS-1)
  const uint32_t rank = crank & 1u;                                 // position in the CTA pair, 0 = leader
  const uint32_t pair = crank >> 1;                                 // pair index inside the cluster (0 .. CS-1)
  const uint32_t leader = pair << 1;                                // cluster rank of this pair's leader
  const int unit = blockIdx.x / (CG * CS);                          // cluster (or CTA) index
  const int n_units = gridDim.x / (CG * CS);
  constexpr int TM = BM * CG;                                       // tile rows
  const int n_tiles_n = p.N / BN;
  const int n_tiles_m = ((p.M + TM - 1) / TM + CS - 1) / CS;        // super-tiles of CS vertically adjacent tiles
  const int n_tiles = n_tiles_m * n_tiles_n;
  const int n_kb = p.K / BK;
  const int n_k4 = p.K / 128;                              // F4C: stages of 256 e2m1 (128 bytes of the K-byte c4 row)
  const int n_steps = PASSES == 2 ? 2 * n_kb : (PASSES == 4 ? n_kb + n_k4 : n_kb);       // ring stages consumed per tile
  // q-th tile of this unit (linear index m * n_tiles_n + n), -1 when the unit is done.
  //   n_inner: the unit walks ALL n-tiles of one m-tile before moving to its next m-tile, so the A tile is re-read
  //            by the same SMs back to back (L2 hits on the same die) instead of by up to n_tiles_n other CTA pairs;
  //   else   : tiles are dealt round-robin, n fastest (neighbouring units share the A tile at the same time).
  auto tile_of = [&](int q) -> int {
    if (p.n_inner) {
      const int mt = unit + (q / n_tiles_n) * n_units;
      return mt < n_tiles_m ? mt * n_tiles_n + q % n_tiles_n : -1;
    }
    const int t = unit + q * n_units;
    return t < n_tiles ? t : -1;
  };

  if (warp == 0 && ptx::elect_one()) {
    ptx::prefetch_tensormap(&tm_a_hi);
    ptx::prefetch_tensormap(&tm_b_hi);
    if (PASSES == 3) {
      ptx::prefetch_tensormap(&tm_a_lo);
      ptx::prefetch_tensormap(&tm_b_lo);
    }
    if (PASSES == 4) {
      ptx::prefetch_tensormap(&tm_a_lo);
      ptx::prefetch_tensormap(&tm_b_lo);
      ptx::prefetch_tensormap(&tm_a_sf);
      ptx::prefetch_tensormap(&tm_b_sf);
    }
    if (EPI == EPI_F32_RED) ptx::prefetch_tensormap(&tm_out);
  }
  if (warp == 1 && ptx::elect_one()) {
    for (int s = 0; s < C::kStages; ++s) {
      ptx::mbar_init(&bars->full[s], 1);
      ptx::mbar_init(&bars->empty[s], CS);                      // every pair of the cluster releases the stage
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&bars->tmem_full[a], 1);
      ptx::mbar_init(&bars->tmem_empty[a], EW * CG);            // leader's copy collects both CTAs' warps
      ptx::mbar_init(&bars->sf_free[a], 4 * CG);                // the four warps (one per lane quadrant) owning columns 0..31
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    if (CG == 2) ptx::tmem_alloc_cg2<C::kTmemCols>(&bars->tmem_base);
    else ptx::tmem_alloc<C::kTmemCols>(&bars->tmem_base);
  }
  if (kGelu4 || EPI == EPI_F32_EMIT) {           // N <= 1024 (checked by the launcher)
    for (int i = threadIdx.x; i < p.N; i += blockDim.x) {
      sm_bias[i] = p.bias[i];
      if (EPI == EPI_GELU_DLN) sm_colsum[i] = p.ln_colsum[i];
    }
  }
  ptx::tc_fence_before();
  if (CG == 2) ptx::cluster_sync(); else __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;
  // EW == 16: 640 threads launch with 96 registers each; the producer warpgroup (warps 0..3) hands its surplus to the
  // epilogue warpgroups.  The setmaxnreg sits INSIDE each role branch: ptxas allocates per branch only then.
#define D3D_PRODUCER_REGS() \
  do { if (EW == 16) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kProducerRegs)); } while (0)

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (both CTAs of a pair)
    D3D_PRODUCER_REGS();
    if (ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      const uint64_t pol_a = ptx::make_l2_policy(p.hint_a), pol_b = ptx::make_l2_policy(p.hint_b);
      for (int q_ = 0, tile; (tile = tile_of(q_)) >= 0; ++q_) {
        const int m0 = ((tile / n_tiles_n) * CS + static_cast<int>(pair)) * TM + static_cast<int>(rank) * BM;
        const int n0 = (tile % n_tiles_n) * BN + static_cast<int>(rank) * C::kBRows;
        int m0_next = -1;                      // first row of this CTA in the unit's next m-tile (n-inner order only)
        if (PASSES == 4 && p.n_inner) {
          const int tn = tile_of(q_ + n_tiles_n - tile % n_tiles_n);      // first tile of the unit's next m-tile
          if (tn >= 0) m0_next = ((tn / n_tiles_n) * CS + static_cast<int>(pair)) * TM + static_cast<int>(rank) * BM;
          if (m0_next >= p.M) m0_next = -1;
        }
        for (int kb = 0; kb < n_steps; ++kb) {
          ptx::mbar_wait(&bars->empty[stage], phase ^ 1);
          uint8_t* s = smem + stage * C::kStageBytes;
          if (PASSES == 4) {
            // fp16 (hi) stages first, then e2m1 (c4) stages with their scale-factor atoms; all bytes of both CTAs complete
            // on the leader's full barrier
            const bool f4 = kb >= n_kb;
            if (p.prefetch_a && m0_next >= 0 && tile % n_tiles_n == (p.prefetch_a == 2 ? n_tiles_n - 1 : 0)) {
              // The A rows of this unit's NEXT m-tile still sit in HBM (an activation operand is 3.3 GB, the L2 126 MB); its
              // first n-tile would wait for them with only the ring's depth of cover.  Pull stage kb of it into L2 now,
              // one whole m-tile ahead (the other n-tiles re-read the rows from L2 anyway).
              const int pc0 = f4 ? (kb - n_kb) * 128 : kb * BK;
              ptx::tma_prefetch_l2_2d(f4 ? &tm_a_lo : &tm_a_hi, pc0, m0_next);
              if (f4) ptx::tma_prefetch_l2_2d(&tm_a_sf, 0, 2 * ((m0_next >> 7) * (p.K / 64) + 2 * (kb - n_kb)));
            }
            const uint32_t full_leader = ptx::mapa(ptx::smem_u32(&bars->full[stage]), leader);
            if (rank == 0)
              ptx::mbar_arrive_expect_tx(&bars->full[stage], 2 * (kTileBytesA + C::kTileBytesB + (f4 ? C::kSfBytes : 0)));
            const int c0 = f4 ? (kb - n_kb) * 128 : kb * BK;      // element coordinate (bytes for the uint8 c4 maps)
            ptx::tma_load_2d_cg2_hint(s, f4 ? &tm_a_lo : &tm_a_hi, full_leader, c0, m0, pol_a);
            ptx::tma_load_2d_cg2_hint(s + kTileBytesA, f4 ? &tm_b_lo : &tm_b_hi, full_leader, c0, n0, pol_b);
            if (f4) {
              // sf arrays viewed as [bytes / 256][256]: an atom (128 rows x 4 k-blocks) is 2 rows, a stage needs the two
              // k-atoms (2 j, 2 j + 1) of a 128-row tile = 4 consecutive rows = 1 KB
              const int apt = p.K / 64;                           // atoms per 128-row tile
              const int ka = 2 * (kb - n_kb);
              uint8_t* sfs = s + kTileBytesA + C::kTileBytesB;
              ptx::tma_load_2d_cg2(sfs, &tm_a_sf, full_leader, 0, 2 * ((m0 >> 7) * apt + ka));
              const int nt0 = ((tile % n_tiles_n) * BN) >> 7;     // first of the two weight row tiles of this n-tile
              ptx::tma_load_2d_cg2(sfs + 1024, &tm_b_sf, full_leader, 0, 2 * (nt0 * apt + ka));
              ptx::tma_load_2d_cg2(sfs + 2048, &tm_b_sf, full_leader, 0, 2 * ((nt0 + 1) * apt + ka));
            }
          } else if (PASSES == 2) {
            // uniform stage: one A tile + one B tile of 128-byte rows; fp16 (hi) stages first, then e5m2 (c8) stages
            const bool f8 = kb >= n_kb;
            const CUtensorMap* ma = f8 ? &tm_a_lo : &tm_a_hi;
            const CUtensorMap* mb = f8 ? &tm_b_lo : &tm_b_hi;
            const int c0 = f8 ? (kb - n_kb) * 128 : kb * BK;      // element coordinate (bytes for the uint8 maps)
            if (CG == 1) {
              ptx::mbar_arrive_expect_tx(&bars->full[stage], C::kStageBytes);
              ptx::tma_load_2d(s, ma, &bars->full[stage], c0, m0);
#pragma unroll
              for (int h = 0; h < C::kBRows / 128; ++h)
                ptx::tma_load_2d(s + kTileBytesA + h * (128 * BK * 2), mb, &bars->full[stage], c0, n0 + h * 128);
            } else {
              const uint32_t full_leader = ptx::mapa(ptx::smem_u32(&bars->full[stage]), leader);
              if (rank == 0) ptx::mbar_arrive_expect_tx(&bars->full[stage], 2 * C::kStageBytes);
              ptx::tma_load_2d_cg2_hint(s, ma, full_leader, c0, m0, pol_a);
              if (CS == 1) {
                ptx::tma_load_2d_cg2_hint(s + kTileBytesA, mb, full_leader, c0, n0, pol_b);
              } else {
                // my 64-row slice of the 128-row weight tile, multicast to the CTA at my position in every pair
                // (the weight maps passed to this instantiation have {128 B x 64 row} boxes)
                constexpr int kSlice = C::kTileBytesB / CS;
                const uint16_t mask = static_cast<uint16_t>((1u << rank) | (1u << (rank + 2)));
                ptx::tma_load_2d_cg2_mc(s + kTileBytesA + pair * kSlice, mb, &bars->full[stage], c0,
                                        n0 + static_cast<int>(pair) * (C::kBRows / CS), mask);
              }
            }
          } else if (CG == 1) {
            ptx::mbar_arrive_expect_tx(&bars->full[stage], C::kStageBytes);
            ptx::tma_load_2d(s, &tm_a_hi, &bars->full[stage], kb * BK, m0);
            s += kTileBytesA;
            if (PASSES == 3) {
              ptx::tma_load_2d(s, &tm_a_lo, &bars->full[stage], kb * BK, m0);
              s += kTileBytesA;
            }
#pragma unroll
            for (int h = 0; h < C::kBRows / 128; ++h)
              ptx::tma_load_2d(s + h * (128 * BK * 2), &tm_b_hi, &bars->full[stage], kb * BK, n0 + h * 128);
            s += C::kTileBytesB;
            if (PASSES == 3) {
#pragma unroll
              for (int h = 0; h < C::kBRows / 128; ++h)
                ptx::tma_load_2d(s + h * (128 * BK * 2), &tm_b_lo, &bars->full[stage], kb * BK, n0 + h * 128);
            }
          } else {
            // both CTAs' bytes complete on the LEADER's full barrier; the leader arms it with the pair's total
            const uint32_t full_leader = ptx::mapa(ptx::smem_u32(&bars->full[stage]), leader);
            if (rank == 0) ptx::mbar_arrive_expect_tx(&bars->full[stage], 2 * C::kStageBytes);
            ptx::tma_load_2d_cg2(s, &tm_a_hi, full_leader, kb * BK, m0);
            s += kTileBytesA;
            if (PASSES == 3) {
              ptx::tma_load_2d_cg2(s, &tm_a_lo, full_leader, kb * BK, m0);
              s += kTileBytesA;
            }
            ptx::tma_load_2d_cg2(s, &tm_b_hi, full_leader, kb * BK, n0);
            s += C::kTileBytesB;
            if (PASSES == 3) ptx::tma_load_2d_cg2(s, &tm_b_lo, full_leader, kb * BK, n0);
          }
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (leader CTA only)
    D3D_PRODUCER_REGS();
    if (rank == 0 && ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::make_idesc_f16(TM, BN, 0 /*fp16*/);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int q_ = 0, tile; (tile = tile_of(q_)) >= 0; ++q_) {
        ptx::mbar_wait(&bars->tmem_empty[acc], acc_phase ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < n_steps; ++kb) {
          ptx::mbar_wait(&bars->full[stage], phase);
          ptx::tc_fence_after();
          const uint32_t s = ptx::smem_u32(smem + stage * C::kStageBytes);
          if (PASSES == 4) {
            if (kb < n_kb) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                ptx::mma_f16_ss_cg2(d_tmem, ptx::make_desc_k_sw128(s + k * 32), ptx::make_desc_k_sw128(s + kTileBytesA + k * 32),
                                    idesc, (kb | k) != 0 ? 1u : 0u);
            } else {
              // scale factors of this stage: smem -> the first 24 columns of the OTHER accumulator (SFA 8 + SFB 16).
              // The previous tile's epilogue has read those columns long before the fp16 stages of this tile are through;
              // sf_free makes it a guarantee.  tcgen05.cp and tcgen05.mma of one thread execute in issue order, so the
              // columns can be rewritten every stage without a wait.
              const uint32_t sf_tmem = tmem_base + (acc ^ 1) * BN;
              if (kb == n_kb && q_ > 0) {
                ptx::mbar_wait(&bars->sf_free[acc ^ 1], ((q_ - 1) >> 1) & 1);
                ptx::tc_fence_after();
              }
              const uint32_t sfs = s + kTileBytesA + C::kTileBytesB;
#pragma unroll
              for (int a = 0; a < 2; ++a) {
                ptx::utccp_32x128b_cg2(sf_tmem + 4 * a, ptx::make_desc_sf(sfs + 512 * a));                  // SFA, k-atom a
                ptx::utccp_32x128b_cg2(sf_tmem + 8 + 8 * a, ptx::make_desc_sf(sfs + 1024 + 512 * a));       // SFB rows 0..127
                ptx::utccp_32x128b_cg2(sf_tmem + 8 + 8 * a + 4, ptx::make_desc_sf(sfs + 2048 + 512 * a));   // SFB rows 128..255
              }
#pragma unroll
              for (int k = 0; k < 4; ++k) {       // 4 x 32 bytes = 4 x 64 e2m1 of K; k-blocks (2k, 2k+1) = bytes 2(k&1).. of atom k>>1
                const uint32_t id4 = ptx::make_idesc_mxf4(TM, BN, (k & 1) * 2);
                ptx::mma_mxf4_ss_cg2(d_tmem, ptx::make_desc_k_sw128(s + k * 32), ptx::make_desc_k_sw128(s + kTileBytesA + k * 32),
                                     id4, sf_tmem + 4 * (k >> 1), sf_tmem + 8 + 8 * (k >> 1), 1u);
              }
            }
            ptx::mma_commit_cg2(&bars->empty[stage], 3);
            if (++stage == C::kStages) { stage = 0; phase ^= 1; }
            continue;
          }
          if (PASSES == 2) {
            constexpr uint32_t idesc8 = ptx::make_idesc_f16(TM, BN, 1 /*e5m2*/);
            const bool f8 = kb >= n_kb;
#pragma unroll
            for (int k = 0; k < 4; ++k) {       // 4 x 32 bytes of K per 128-byte row: K = 16 (fp16) or 32 (e5m2)
              const uint64_t da = ptx::make_desc_k_sw128(s + k * 32);
              const uint64_t db = ptx::make_desc_k_sw128(s + kTileBytesA + k * 32);
              const uint32_t accum = (kb | k) != 0 ? 1u : 0u;
              if (f8) {
                if (CG == 2) ptx::mma_f8_ss_cg2(d_tmem, da, db, idesc8, accum);
                else ptx::mma_f8_ss(d_tmem, da, db, idesc8, accum);
              } else {
                if (CG == 2) ptx::mma_f16_ss_cg2(d_tmem, da, db, idesc, accum);
                else ptx::mma_f16_ss(d_tmem, da, db, idesc, accum);
              }
            }
            // frees the stage: in both CTAs of this pair and (CS == 2) in the pair that multicasts into them
            if (CG == 2) ptx::mma_commit_cg2(&bars->empty[stage], static_cast<uint16_t>((1u << (2 * CS)) - 1));
            else ptx::mma_commit(&bars->empty[stage]);
            if (++stage == C::kStages) { stage = 0; phase ^= 1; }
            continue;
          }
          const uint32_t a_hi = s;
          const uint32_t a_lo = s + kTileBytesA;
          const uint32_t b_hi = s + (PASSES == 3 ? 2 : 1) * kTileBytesA;
          const uint32_t b_lo = b_hi + C::kTileBytesB;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint64_t da_hi = ptx::make_desc_k_sw128(a_hi + k * 32);
            const uint64_t db_hi = ptx::make_desc_k_sw128(b_hi + k * 32);
            const uint32_t accum = (kb | k) != 0 ? 1u : 0u;
            if (CG == 2) ptx::mma_f16_ss_cg2(d_tmem, da_hi, db_hi, idesc, accum);
            else ptx::mma_f16_ss(d_tmem, da_hi, db_hi, idesc, accum);
            if (PASSES == 3) {
              const uint64_t da_lo = ptx::make_desc_k_sw128(a_lo + k * 32);
              const uint64_t db_lo = ptx::make_desc_k_sw128(b_lo + k * 32);
              if (CG == 2) {
                ptx::mma_f16_ss_cg2(d_tmem, da_hi, db_lo, idesc, 1u);
                ptx::mma_f16_ss_cg2(d_tmem, da_lo, db_hi, idesc, 1u);
              } else {
                ptx::mma_f16_ss(d_tmem, da_hi, db_lo, idesc, 1u);
                ptx::mma_f16_ss(d_tmem, da_lo, db_hi, idesc, 1u);
              }
            }
          }
          // frees the smem stage (in both CTAs) once these MMAs have read it
          if (CG == 2) ptx::mma_commit_cg2(&bars->empty[stage], 3);
          else ptx::mma_commit(&bars->empty[stage]);
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
        // accumulator complete -> epilogue warps (of both CTAs of this pair)
        if (CG == 2) ptx::mma_commit_cg2(&bars->tmem_full[acc], static_cast<uint16_t>(3u << leader));
        else ptx::mma_commit(&bars->tmem_full[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp < 4) {
    D3D_PRODUCER_REGS();
  } else {
    // ------------------------------------------------------------ epilogue (EW warps per CTA)
    if (EW == 16) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kEpilogueRegs));
    // TMEM hands every lane one ROW (32 consecutive columns); storing that layout directly costs 32 cache lines
    // per store instruction and made the epilogue, not the MMA, the bottleneck (1-pass and 3-pass GEMMs took
    // the same time).  Each warp therefore transposes its 32 x 32 chunk through a swizzled 4 KB buffer and
    // moves global data with "8 lanes = 128 contiguous bytes of one row" accesses (4 rows per instruction).
    const int q = warp & 3;                 // TMEM lane quadrant this warp may access
    const int half = (warp - 4) >> 2;       // which slice of the BN columns (BN / kColsW columns each)
    constexpr int kColsW = BN / (EW / 4);   // columns per warp
    constexpr int kChunks = kColsW / 32;    // 32-column chunks per warp
    const uint32_t stg = ptx::smem_u32(staging) + (warp - 4) * 4096;
    const int rsub = lane >> 3, gsub = lane & 7;      // coalesced mapping: instruction j covers rows 4j + rsub
    int acc = 0;
    uint32_t acc_phase = 0;
    // EPI_F32_LN: running (mean, M2) of this lane's row over the 128 columns this warp owns in each accumulator
    float ln_mean[2] = {0.f, 0.f}, ln_m2[2] = {0.f, 0.f};
    constexpr bool kSmemVec = kGelu4 || EPI == EPI_F32_EMIT;     // bias / column sums come from shared memory
    const F4cStore f4st = EPI == EPI_F32_EMIT ? f4c_store_init(p.emit_hi, p.emit_c4, p.N, gsub)
                                              : f4c_store_init(p.out_hi, reinterpret_cast<uint8_t*>(p.out_lo), p.N, gsub);
    // PASSES == 4 (the shipped kernel): streaming stores are compiled in (D3D_GEMM_STREAM_OUT=0 at BUILD time for the A/B);
    // a run-time choice cost two predicated stores and four R2UR per store instruction (distinct memory descriptors)
#ifndef D3D_GEMM_STREAM_OUT
#define D3D_GEMM_STREAM_OUT 1
#endif
    const bool stream_out = PASSES == 4 ? (D3D_GEMM_STREAM_OUT != 0) : (p.stream_out != 0);
    // EPI_GELU_DLN: (rstd, -rstd mean) of this lane's row, valid for all n-tiles of the current m-tile; the partial sums
    // of the NEXT m-tile's row are fetched a few per tile while this m-tile is processed (their latency would otherwise
    // sit on the epilogue's critical path, which sets the tile time of fc1)
    ptx::f32x2 dln_a = ptx::splat2(1.0f), dln_b = ptx::splat2(0.0f);
    int dln_mt = -1;                         // m-tile the pair (dln_a, dln_b) belongs to
    float dln_s1 = 0.f, dln_s2 = 0.f;        // sums gathered so far for m-tile dln_next_mt
    int dln_next_mt = -1, dln_parts_done = 0;
    auto dln_row_of = [&](int mt) { return ((mt * CS + static_cast<int>(pair)) * TM + static_cast<int>(rank) * BM) + q * 32 + lane; };
    for (int q_ = 0, tile; (tile = tile_of(q_)) >= 0; ++q_) {
      const int m0 = ((tile / n_tiles_n) * CS + static_cast<int>(pair)) * TM + static_cast<int>(rank) * BM;
      const int n0 = (tile % n_tiles_n) * BN;
      const int row_w = m0 + q * 32;                    // first row of this warp
      const int colbase = n0 + half * kColsW;
      const bool has_res = kF32 && p.residual != nullptr;
      // Residual prefetch, kResDepth chunks deep (registers).  The fp32 + residual epilogue moves 256 KB per CTA and tile
      // (read + write) and, with the F4C mainloop at ~5 us per tile, sets the tile time of proj / fc2: ncu had them at
      // 55-58 % of DRAM with ONE 4 KB chunk per warp in flight (32 KB per SM, below bandwidth x latency ~ 44 B/ns x 0.8 us);
      // two chunks per warp double the bytes in flight (profiles/r02d_full_gemm.md -> r02e).
      constexpr int kResDepth = (EPI == EPI_F32 && EW == 8) ? D3D_GEMM_RES_DEPTH : 1;      // EMIT / 16 warps: no registers to spare
      // 16 warps at 104 registers: x (32 registers) stays live through the operand emission, so the next residual chunk is
      // requested only after it (four warps per scheduler cover the exposed latency)
      constexpr bool kLateRes = EPI == EPI_F32_EMIT && EW == 16;
      float4 resv[kResDepth][8];
      auto load_res = [&](int ci) {                     // residual chunk ci, coalesced (row 4j + rsub, granule gsub)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int rr = row_w + 4 * j + rsub;
          const float* src = p.residual + static_cast<size_t>(rr) * p.N + colbase + ci * 32 + gsub * 4;
          resv[ci % kResDepth][j] = rr >= p.M ? make_float4(0.f, 0.f, 0.f, 0.f)
                                              : (stream_out ? ptx::ld_global_cs(src) : *reinterpret_cast<const float4*>(src));
        }
      };
      if (has_res) {                         // in flight while the accumulator is still being computed
#pragma unroll
        for (int c = 0; c < kResDepth; ++c) load_res(c);
      }
      uint32_t sfp_w = 0, sfq_w = 0;         // F4C output operand: this row's scale bytes of the tile's k-blocks (P / Q part)
      ptx::f32x2 ln_s1p = ptx::splat2(0.f), ln_s2p = ptx::splat2(0.f);   // EPI_F32_EMIT: (sum, sum of squares) of this lane's row, 64 columns
      float2 dln_pf[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};   // partial sums in flight during this tile
      int dln_pf_n = 0;
      if (EPI == EPI_GELU_DLN) {
        const int parts = p.K >> 6;
        const int mt = tile / n_tiles_n;
        if (mt != dln_mt) {
          // statistics of this m-tile: whatever was not prefetched is loaded now (all of it for the first m-tile)
          const int rr = dln_row_of(mt);
          if (dln_next_mt != mt) { dln_s1 = 0.f; dln_s2 = 0.f; dln_parts_done = 0; }
          if (rr < p.M)           // same order of additions as the prefetched path: results must not depend on which
            for (int pt = dln_parts_done; pt < parts; pt += 2) {      // tiles of a CTA a row falls into (batch-split invariance)
              const float2 v0 = p.ln_stats[static_cast<size_t>(pt) * p.M + rr];
              const float2 v1 = p.ln_stats[static_cast<size_t>(pt + 1) * p.M + rr];
              dln_s1 += v0.x + v1.x; dln_s2 += v0.y + v1.y;
            }
          const float inv_k = 1.0f / static_cast<float>(p.K);
          const float mean = dln_s1 * inv_k;
          const float var = fmaxf(fmaf(-mean, mean, dln_s2 * inv_k), 0.0f);
          const float rstd = 1.0f / sqrtf(var + p.ln_eps);
          dln_a = ptx::splat2(rstd);
          dln_b = ptx::splat2(-rstd * mean);
          dln_mt = mt;
          dln_s1 = 0.f; dln_s2 = 0.f; dln_parts_done = 0;
          const int nt = tile_of(q_ + n_tiles_n - tile % n_tiles_n);       // first tile of this unit's next m-tile
          dln_next_mt = nt >= 0 ? nt / n_tiles_n : -1;
        }
        if (dln_next_mt >= 0 && dln_parts_done < parts) {                   // two more parts of the next m-tile's row
          const int rr = dln_row_of(dln_next_mt);
          dln_pf_n = 2;                                                     // K % 128 == 0: an even number of parts
          if (rr < p.M) {
            dln_pf[0] = p.ln_stats[static_cast<size_t>(dln_parts_done) * p.M + rr];
            dln_pf[1] = p.ln_stats[static_cast<size_t>(dln_parts_done + 1) * p.M + rr];
          }
        }
      }
      ptx::mbar_wait(&bars->tmem_full[acc], acc_phase);
      ptx::tc_fence_after();
#pragma unroll
      for (int ci = 0; ci < kChunks; ++ci) {
        const int col0 = half * kColsW + ci * 32;       // column inside the tile
        uint32_t r[32];
        ptx::tmem_ld_32x32(tmem_base + acc * BN + col0 + (static_cast<uint32_t>(q * 32) << 16), r);
        if (has_res) {
#pragma unroll
          for (int j = 0; j < 8; ++j) stg_st(stg, 4 * j + rsub, gsub, *reinterpret_cast<uint4*>(&resv[ci % kResDepth][j]));
          __syncwarp();
          if (!kLateRes && ci + kResDepth < kChunks) load_res(ci + kResDepth);
        }
        const int gcol = n0 + col0;
        float4 bias4[8];                                 // issued before the TMEM wait so their latency is hidden
        if (!kSmemVec) {
#pragma unroll
          for (int v = 0; v < 8; ++v) bias4[v] = __ldg(reinterpret_cast<const float4*>(p.bias + gcol) + v);
        }
        const uint32_t sb4 = ptx::smem_u32(sm_bias + gcol), sc4 = ptx::smem_u32(sm_colsum + gcol);   // kSmemVec: read just in time
        ptx::tmem_ld_wait();
        if (PASSES == 4 && ci == 0 && half == 0) {
          // columns 0..31 of this accumulator are in registers: the NEXT tile's e2m1 stages may put their scale factors there
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&bars->sf_free[acc]), leader));
        }
        if (EPI == EPI_F32_RED) {
          // X += acc + bias: the chunk goes into the staging buffer (lane = row; the buffer's swizzle is the tensor map's
          // SWIZZLE_128B) and one lane hands it to the TMA unit as an fp32 add-reduction into X.  The buffer is reused once
          // the previous reduction has READ it (bulk async-group).
          if (lane == 0) ptx::bulk_wait_read_all();
          __syncwarp();
#pragma unroll
          for (int v = 0; v < 8; ++v) {
            const float4 b = bias4[v];
            stg_st(stg, lane, v, make_uint4(__float_as_uint(__uint_as_float(r[4 * v + 0]) + b.x), __float_as_uint(__uint_as_float(r[4 * v + 1]) + b.y),
                                            __float_as_uint(__uint_as_float(r[4 * v + 2]) + b.z), __float_as_uint(__uint_as_float(r[4 * v + 3]) + b.w)));
          }
          ptx::fence_proxy_async();            // generic-proxy writes -> visible to the async proxy (TMA)
          __syncwarp();
          if (lane == 0) {
            ptx::tma_reduce_add_2d(&tm_out, stg, gcol, row_w);
            ptx::bulk_commit();
          }
        } else if (EPI == EPI_F32_EMIT) {
          // x = acc + bias + residual on packed pairs; x stays in r for the operand image; (sum, sum of squares) per lane
#pragma unroll
          for (int v = 0; v < 8; ++v) {
            const float4 b = lds_f4(sb4 + 16 * v);
            const uint4 ru = stg_ld(stg, lane, v);
            const ptx::f32x2 o01 = ptx::add2(ptx::add2(ptx::pack2(__uint_as_float(r[4 * v + 0]), __uint_as_float(r[4 * v + 1])), ptx::pack2(b.x, b.y)),
                                             ptx::pack2(__uint_as_float(ru.x), __uint_as_float(ru.y)));
            const ptx::f32x2 o23 = ptx::add2(ptx::add2(ptx::pack2(__uint_as_float(r[4 * v + 2]), __uint_as_float(r[4 * v + 3])), ptx::pack2(b.z, b.w)),
                                             ptx::pack2(__uint_as_float(ru.z), __uint_as_float(ru.w)));
            float o0, o1, o2, o3;
            ptx::unpack2(o01, o0, o1);
            ptx::unpack2(o23, o2, o3);
            r[4 * v + 0] = __float_as_uint(o0); r[4 * v + 1] = __float_as_uint(o1);
            r[4 * v + 2] = __float_as_uint(o2); r[4 * v + 3] = __float_as_uint(o3);
            stg_st(stg, lane, v, make_uint4(r[4 * v + 0], r[4 * v + 1], r[4 * v + 2], r[4 * v + 3]));
            ln_s1p = ptx::add2(ln_s1p, ptx::add2(o01, o23));
            ln_s2p = ptx::fma2(o01, o01, ptx::fma2(o23, o23, ln_s2p));
          }
          __syncwarp();
          uint4 vals[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) vals[j] = stg_ld(stg, 4 * j + rsub, gsub);
          {
            float* d = p.out_f32 + static_cast<size_t>(row_w + rsub) * p.N + gcol + gsub * 4;
            const size_t step = static_cast<size_t>(4) * p.N;
            if (p.M - row_w >= 32) {
#pragma unroll
              for (int j = 0; j < 8; ++j) { ptx::st_global_cs(d, vals[j]); d += step; }
            } else {
#pragma unroll
              for (int j = 0; j < 8; ++j) { if (row_w + 4 * j + rsub < p.M) ptx::st_global_cs(d, vals[j]); d += step; }
            }
          }
          __syncwarp();                        // every lane has read the fp32 rows out of the staging buffer
          f4c_emit_chunk(r, stg, lane, row_w, gcol, p.M, f4st, stream_out, sfp_w, sfq_w);
          if (kLateRes && ci + 1 < kChunks) load_res(ci + 1);
          if (ci & 1) {                        // two chunks = 64 columns = one statistics part
            const int rr = row_w + lane;
            float a0, a1, q0, q1;
            ptx::unpack2(ln_s1p, a0, a1);
            ptx::unpack2(ln_s2p, q0, q1);
            if (rr < p.M) p.ln_stats[static_cast<size_t>(gcol >> 6) * p.M + rr] = make_float2(a0 + a1, q0 + q1);
            ln_s1p = ptx::splat2(0.f); ln_s2p = ptx::splat2(0.f);
          }
        } else if (kF32) {
          float csum = 0.f;
#pragma unroll
          for (int v = 0; v < 8; ++v) {
            const float4 b = kSmemVec ? lds_f4(sb4 + 16 * v) : bias4[v];
            float4 o;
            o.x = __uint_as_float(r[4 * v + 0]) + b.x;
            o.y = __uint_as_float(r[4 * v + 1]) + b.y;
            o.z = __uint_as_float(r[4 * v + 2]) + b.z;
            o.w = __uint_as_float(r[4 * v + 3]) + b.w;
            if (has_res) {
              const uint4 ru = stg_ld(stg, lane, v);
              o.x += __uint_as_float(ru.x); o.y += __uint_as_float(ru.y); o.z += __uint_as_float(ru.z); o.w += __uint_as_float(ru.w);
            }
            stg_st(stg, lane, v, make_uint4(__float_as_uint(o.x), __float_as_uint(o.y), __float_as_uint(o.z), __float_as_uint(o.w)));
            if (EPI == EPI_F32_LN) {           // keep x for the statistics and the TMEM write-back
              r[4 * v + 0] = __float_as_uint(o.x); r[4 * v + 1] = __float_as_uint(o.y);
              r[4 * v + 2] = __float_as_uint(o.z); r[4 * v + 3] = __float_as_uint(o.w);
              csum += (o.x + o.y) + (o.z + o.w);
            }
          }
          if (EPI == EPI_F32_LN) {
            // x goes back into the accumulator columns (pass 2 normalises it without re-reading the residual), and the
            // chunk's (mean, M2) joins the lane's running pair (Chan et al.: no E[x^2] - mean^2 cancellation)
            ptx::tmem_st_32x32(tmem_base + acc * BN + col0 + (static_cast<uint32_t>(q * 32) << 16), r);
            const float cmean = csum * (1.0f / 32.0f);
            float cm2 = 0.f;
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              const float d = __uint_as_float(r[e]) - cmean;
              cm2 = fmaf(d, d, cm2);
            }
            const float cnt = 32.0f * ci, tot = cnt + 32.0f;
            const float delta = cmean - ln_mean[acc];
            if (ci == 0) { ln_mean[acc] = cmean; ln_m2[acc] = cm2; }
            else {
              ln_mean[acc] += delta * (32.0f / tot);
              ln_m2[acc] += cm2 + delta * delta * (cnt * 32.0f / tot);
            }
          }
          __syncwarp();
          uint4 vals[8];                       // all shared loads first, then all global stores (distinct registers)
#pragma unroll
          for (int j = 0; j < 8; ++j) vals[j] = stg_ld(stg, 4 * j + rsub, gsub);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int rr = row_w + 4 * j + rsub;
            if (rr < p.M) {
              float* dst = p.out_f32 + static_cast<size_t>(rr) * p.N + gcol + gsub * 4;
              if (stream_out) ptx::st_global_cs(dst, vals[j]); else *reinterpret_cast<uint4*>(dst) = vals[j];
            }
          }
        } else if (kGelu4) {
          // FMT_F4C operand of fc2: this lane's 32 columns are exactly one scale block of each part.  Pass 1: GELU, hi
          // halves into the staging row (granules 0..3), block maxima of x and of x - hi; pass 2: both e2m1 images
          // (granule 4 = 32 nibbles of P = q4(x), granule 5 = Q = q4(x - hi)); the two scale bytes join the lane's words.
          float ax = 0.f, al = 0.f;
#pragma unroll
          for (int v = 0; v < 4; ++v) {
            uint32_t hw[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float4 b = lds_f4(sb4 + 16 * (2 * v + (e >> 1)));
              const ptx::f32x2 accp = ptx::pack2(__uint_as_float(r[8 * v + 2 * e + 0]), __uint_as_float(r[8 * v + 2 * e + 1]));
              ptx::f32x2 bp2 = (e & 1) ? ptx::pack2(b.z, b.w) : ptx::pack2(b.x, b.y);
              ptx::f32x2 xp;
              if (EPI == EPI_GELU_DLN) {        // rstd acc + (c_n - rstd mean s_n)
                const float4 cs = lds_f4(sc4 + 16 * (2 * v + (e >> 1)));
                bp2 = ptx::fma2(dln_b, (e & 1) ? ptx::pack2(cs.z, cs.w) : ptx::pack2(cs.x, cs.y), bp2);
                xp = ptx::fma2(dln_a, accp, bp2);
              } else {
                xp = ptx::add2(accp, bp2);
              }
              xp = gelu_erf2(xp);
              float x0, x1;
              ptx::unpack2(xp, x0, x1);
              const __half2 h01 = __floats2half2_rn(x0, x1);
              const float2 hf = __half22float2(h01);
              hw[e] = *reinterpret_cast<const uint32_t*>(&h01);
              ax = fmaxf(ax, fmaxf(fabsf(x0), fabsf(x1)));
              al = fmaxf(al, fmaxf(fabsf(x0 - hf.x), fabsf(x1 - hf.y)));
              r[8 * v + 2 * e + 0] = __float_as_uint(x0);
              r[8 * v + 2 * e + 1] = __float_as_uint(x1);
            }
            stg_st(stg, lane, v, make_uint4(hw[0], hw[1], hw[2], hw[3]));
          }
          const uint32_t bp = op_ue8m0_of(ax), bq = op_ue8m0_of(al);
          const ptx::f32x2 ip = ptx::splat2(op_ue8m0_inv(bp)), iq = ptx::splat2(op_ue8m0_inv(bq));
          uint32_t pw[4], qw[4];
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            uint32_t pa = 0, qa = 0;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float x0 = __uint_as_float(r[8 * w + 2 * e + 0]), x1 = __uint_as_float(r[8 * w + 2 * e + 1]);
              const float2 hf = __half22float2(__floats2half2_rn(x0, x1));
              float a0, a1, l0, l1;
              ptx::unpack2(ptx::mul2(ptx::pack2(x0, x1), ip), a0, a1);
              ptx::unpack2(ptx::mul2(ptx::sub2(ptx::pack2(x0, x1), ptx::pack2(hf.x, hf.y)), iq), l0, l1);
              pa |= op_e2m1x2(a0, a1) << (8 * e);
              qa |= op_e2m1x2(l0, l1) << (8 * e);
            }
            pw[w] = pa; qw[w] = qa;
          }
          stg_st(stg, lane, 4, make_uint4(pw[0], pw[1], pw[2], pw[3]));
          stg_st(stg, lane, 5, make_uint4(qw[0], qw[1], qw[2], qw[3]));
          sfp_w |= bp << (8 * ((gcol >> 5) & 3));
          sfq_w |= bq << (8 * ((gcol >> 5) & 3));
          __syncwarp();
          f4c_store_chunk(f4st, stg, rsub, gsub, row_w, gcol, p.M, stream_out);
        } else {
          // fp16 outputs: row = hi (granules 0..3, 32 halves) | second part (granules 4..7):
          //   fp16 lo (FMT_SPLIT16, and always for q|k|v), or for the FMT_F8C fc2 operand
          //   granules 4,5 = e5m2(x 2^-8) and 6,7 = e5m2(lo 2^4) of the 32 columns
          constexpr bool gelu = EPI == EPI_GELU_SPLIT;
          constexpr bool f8out = EPI == EPI_GELU_SPLIT && PASSES == 2;
          uint32_t a8w[8], l8w[8];
#pragma unroll
          for (int v = 0; v < 4; ++v) {
            uint32_t hw[4], lw[4], a16[4], l16[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float4 b = bias4[2 * v + (e >> 1)];
#if D3D_EPI_PACKED
              ptx::f32x2 xp = ptx::add2(ptx::pack2(__uint_as_float(r[8 * v + 2 * e + 0]), __uint_as_float(r[8 * v + 2 * e + 1])),
                                        (e & 1) ? ptx::pack2(b.z, b.w) : ptx::pack2(b.x, b.y));
              if (gelu) xp = gelu_erf2(xp);
              float x0, x1, l0, l1;
              ptx::unpack2(xp, x0, x1);
              const __half2 h01 = __floats2half2_rn(x0, x1);
              const float2 hf = __half22float2(h01);
              const ptx::f32x2 lp = ptx::sub2(xp, ptx::pack2(hf.x, hf.y));
              ptx::unpack2(lp, l0, l1);
              hw[e] = *reinterpret_cast<const uint32_t*>(&h01);
              if (f8out) {
                ptx::unpack2(ptx::mul2(xp, ptx::splat2(kActHiScale)), x0, x1);
                ptx::unpack2(ptx::mul2(lp, ptx::splat2(kActLoScale)), l0, l1);
                a16[e] = op_e5m2x2(x0, x1);
                l16[e] = op_e5m2x2(l0, l1);
              } else {
                const __half2 l01 = __floats2half2_rn(l0, l1);
                lw[e] = *reinterpret_cast<const uint32_t*>(&l01);
              }
#else
              float x0 = __uint_as_float(r[8 * v + 2 * e + 0]) + ((e & 1) ? b.z : b.x);
              float x1 = __uint_as_float(r[8 * v + 2 * e + 1]) + ((e & 1) ? b.w : b.y);
              if (gelu) { x0 = gelu_erf(x0); x1 = gelu_erf(x1); }
              const __half h0 = __float2half_rn(x0), h1 = __float2half_rn(x1);
              const float l0 = x0 - __half2float(h0), l1 = x1 - __half2float(h1);
              hw[e] = pack_h2(h0, h1);
              if (f8out) {
                a16[e] = op_e5m2x2(x0 * kActHiScale, x1 * kActHiScale);
                l16[e] = op_e5m2x2(l0 * kActLoScale, l1 * kActLoScale);
              } else {
                lw[e] = pack_h2(__float2half_rn(l0), __float2half_rn(l1));
              }
#endif
            }
            stg_st(stg, lane, v, make_uint4(hw[0], hw[1], hw[2], hw[3]));
            if (f8out) {
              a8w[2 * v] = a16[0] | (a16[1] << 16); a8w[2 * v + 1] = a16[2] | (a16[3] << 16);
              l8w[2 * v] = l16[0] | (l16[1] << 16); l8w[2 * v + 1] = l16[2] | (l16[3] << 16);
            } else {
              stg_st(stg, lane, 4 + v, make_uint4(lw[0], lw[1], lw[2], lw[3]));
            }
          }
          if (f8out) {
            stg_st(stg, lane, 4, make_uint4(a8w[0], a8w[1], a8w[2], a8w[3]));
            stg_st(stg, lane, 5, make_uint4(a8w[4], a8w[5], a8w[6], a8w[7]));
            stg_st(stg, lane, 6, make_uint4(l8w[0], l8w[1], l8w[2], l8w[3]));
            stg_st(stg, lane, 7, make_uint4(l8w[4], l8w[5], l8w[6], l8w[7]));
          }
          __syncwarp();
          __half* hi_base;
          __half* lo_base;          // null: this chunk has no lo output (q, k)
          size_t ld;
          if (EPI == EPI_GELU_SPLIT) {
            hi_base = p.out_hi + gcol; lo_base = p.out_lo + gcol; ld = static_cast<size_t>(p.N);
          } else {                   // EPI_QKV16: q | k -> fp16; v -> hi at the same column, lo 512 columns further
            hi_base = p.out_qkv + gcol; lo_base = gcol >= 2 * kC ? p.out_qkv + gcol + kC : nullptr; ld = kQkvRow;
          }
          if (EPI == EPI_GELU_SPLIT && PASSES == 2) {
            // c8 row of the fc2 operand: N bytes e5m2(x 2^-8) then N bytes e5m2(lo 2^4); 32 columns = 2 granules each
            uint8_t* c8 = reinterpret_cast<uint8_t*>(p.out_lo);
            uint4 vals[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) vals[j] = stg_ld(stg, 4 * j + rsub, gsub);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int rr = row_w + 4 * j + rsub;
              if (rr >= p.M) continue;
              void* dst = gsub < 4 ? static_cast<void*>(p.out_hi + static_cast<size_t>(rr) * p.N + gcol + gsub * 8)
                                   : static_cast<void*>(c8 + static_cast<size_t>(rr) * (2 * p.N) + (gsub < 6 ? 0 : p.N) +
                                                        gcol + (gsub & 1) * 16);
              if (stream_out) ptx::st_global_cs(dst, vals[j]); else *reinterpret_cast<uint4*>(dst) = vals[j];
            }
          } else {
            __half* dst_base = gsub < 4 ? hi_base : lo_base;
            uint4 vals[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) vals[j] = stg_ld(stg, 4 * j + rsub, gsub);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int rr = row_w + 4 * j + rsub;
              if (rr < p.M && dst_base) {
                __half* dst = dst_base + static_cast<size_t>(rr) * ld + (gsub & 3) * 8;
                if (stream_out) ptx::st_global_cs(dst, vals[j]); else *reinterpret_cast<uint4*>(dst) = vals[j];
              }
            }
          }
        }
        __syncwarp();          // the buffer is rewritten by the next chunk
      }
      if (kGelu4 || EPI == EPI_F32_EMIT) {
        // scale bytes of row (row_w + lane): k-blocks colbase/32 .. +kChunks-1 of part P, the same + N/32 of part Q; they
        // are adjacent bytes of one scale-factor atom (operand.cuh), written as one word (4 chunks) or half-word (2)
        const int rr = row_w + lane;
        if (rr < p.M) {
          const int kb0 = colbase >> 5, apt = p.N / 64;
          uint8_t* sf_out = EPI == EPI_F32_EMIT ? p.emit_sf : p.out_sf;
          uint8_t* dp = sf_out + op_sf_offset(rr, kb0, apt);
          uint8_t* dq = sf_out + op_sf_offset(rr, (p.N >> 5) + kb0, apt);
          if (kChunks == 4) {
            *reinterpret_cast<uint32_t*>(dp) = sfp_w;
            *reinterpret_cast<uint32_t*>(dq) = sfq_w;
          } else {
            *reinterpret_cast<uint16_t*>(dp) = static_cast<uint16_t>(sfp_w >> (8 * (kb0 & 3)));
            *reinterpret_cast<uint16_t*>(dq) = static_cast<uint16_t>(sfq_w >> (8 * (kb0 & 3)));
          }
        }
      }
      if (EPI == EPI_F32_LN) {
        // The two n-tiles of a row tile land in accumulators 0 and 1 back to back (n-inner order, N == 2 BN).  After
        // pass 1 of the second one the full 512-wide rows are known: exchange the partial statistics with the warp that
        // owns the other 128 columns of these rows, then pass 2 re-reads x from TMEM, normalises and writes the next
        // GEMM's A operand.  Accumulator 0 is released only here (x lives in it between the passes).
        if (acc == 1) {
          ptx::tmem_st_wait();
          *reinterpret_cast<float4*>(staging + (warp - 4) * 4096 + lane * 16) = make_float4(ln_mean[0], ln_m2[0], ln_mean[1], ln_m2[1]);
          ptx::bar_sync(1, EW * 32);
          const float4 oth = *reinterpret_cast<const float4*>(staging + ((warp - 4) ^ 4) * 4096 + lane * 16);
          ptx::bar_sync(1, EW * 32);                       // every partner row is read: the buffers may be reused
          // Chan combination of equal-sized groups: mean = (a + b) / 2, M2 = M2a + M2b + (b - a)^2 n / 2
          const float d0 = oth.x - ln_mean[0], d1 = oth.z - ln_mean[1];
          const float mean0 = ln_mean[0] + 0.5f * d0, m20 = ln_m2[0] + oth.y + d0 * d0 * 64.0f;     // 256 columns each
          const float mean1 = ln_mean[1] + 0.5f * d1, m21 = ln_m2[1] + oth.w + d1 * d1 * 64.0f;
          const float dd = mean1 - mean0;
          const float mean = mean0 + 0.5f * dd;
          const float var = (m20 + m21 + dd * dd * 128.0f) * (1.0f / 512.0f);
          const float rstd = 1.0f / sqrtf(var + p.ln_eps);      // as ln_rows() of rowwise.cu
          uint8_t* c8 = reinterpret_cast<uint8_t*>(p.ln_second);
#pragma unroll
          for (int a = 0; a < 2; ++a) {
#pragma unroll
            for (int ci = 0; ci < kChunks; ++ci) {
              const int col0 = half * kColsW + ci * 32;
              const int gcol = a * BN + col0;
              uint32_t r[32];
              ptx::tmem_ld_32x32(tmem_base + a * BN + col0 + (static_cast<uint32_t>(q * 32) << 16), r);
              ptx::tmem_ld_wait();
              uint32_t a8w[8], l8w[8];
#pragma unroll
              for (int v = 0; v < 4; ++v) {
                const float4 g0 = __ldg(reinterpret_cast<const float4*>(p.ln_gamma + gcol) + 2 * v);
                const float4 g1 = __ldg(reinterpret_cast<const float4*>(p.ln_gamma + gcol) + 2 * v + 1);
                const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.ln_beta + gcol) + 2 * v);
                const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.ln_beta + gcol) + 2 * v + 1);
                const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
                const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                uint32_t hw[4], a16[4], l16[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float x0 = fmaf((__uint_as_float(r[8 * v + 2 * e]) - mean) * rstd, gg[2 * e], bb[2 * e]);
                  const float x1 = fmaf((__uint_as_float(r[8 * v + 2 * e + 1]) - mean) * rstd, gg[2 * e + 1], bb[2 * e + 1]);
                  const __half h0 = __float2half_rn(x0), h1 = __float2half_rn(x1);
                  hw[e] = pack_h2(h0, h1);
                  a16[e] = op_e5m2x2(x0 * kActHiScale, x1 * kActHiScale);
                  l16[e] = op_e5m2x2((x0 - __half2float(h0)) * kActLoScale, (x1 - __half2float(h1)) * kActLoScale);
                }
                stg_st(stg, lane, v, make_uint4(hw[0], hw[1], hw[2], hw[3]));
                a8w[2 * v] = a16[0] | (a16[1] << 16); a8w[2 * v + 1] = a16[2] | (a16[3] << 16);
                l8w[2 * v] = l16[0] | (l16[1] << 16); l8w[2 * v + 1] = l16[2] | (l16[3] << 16);
              }
              stg_st(stg, lane, 4, make_uint4(a8w[0], a8w[1], a8w[2], a8w[3]));
              stg_st(stg, lane, 5, make_uint4(a8w[4], a8w[5], a8w[6], a8w[7]));
              stg_st(stg, lane, 6, make_uint4(l8w[0], l8w[1], l8w[2], l8w[3]));
              stg_st(stg, lane, 7, make_uint4(l8w[4], l8w[5], l8w[6], l8w[7]));
              __syncwarp();
              uint4 vals[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) vals[j] = stg_ld(stg, 4 * j + rsub, gsub);
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const int rr = row_w + 4 * j + rsub;
                if (rr >= p.M) continue;
                void* dst = gsub < 4 ? static_cast<void*>(p.ln_hi + static_cast<size_t>(rr) * p.N + gcol + gsub * 8)
                                     : static_cast<void*>(c8 + static_cast<size_t>(rr) * (2 * p.N) + (gsub < 6 ? 0 : p.N) +
                                                          gcol + (gsub & 1) * 16);
                if (stream_out) ptx::st_global_cs(dst, vals[j]); else *reinterpret_cast<uint4*>(dst) = vals[j];
              }
              __syncwarp();
            }
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if (CG == 2) ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&bars->tmem_empty[a]), leader));
              else ptx::mbar_arrive(&bars->tmem_empty[a]);
            }
          }
        }
      } else {
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (CG == 2) ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&bars->tmem_empty[acc]), leader));
          else ptx::mbar_arrive(&bars->tmem_empty[acc]);
        }
      }
      if (EPI == EPI_GELU_DLN && dln_pf_n > 0) {       // the prefetched partial sums have long arrived
        dln_s1 += dln_pf[0].x + dln_pf[1].x;
        dln_s2 += dln_pf[0].y + dln_pf[1].y;
        dln_parts_done += dln_pf_n;
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (EPI == EPI_F32_RED && lane == 0) ptx::bulk_wait_all();     // the staging buffer must outlive the last reduction
  }
#undef D3D_PRODUCER_REGS
  __syncwarp();

  ptx::tc_fence_before();
  if (CG == 2) ptx::cluster_sync(); else __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    if (CG == 2) ptx::tmem_dealloc_cg2<C::kTmemCols>(tmem_base);
    else ptx::tmem_dealloc<C::kTmemCols>(tmem_base);
  }
}

// Clusters of 4 cannot straddle a GPC, so fewer than 148/4 of them may be co-resident: ask the runtime.
template <int CG, int BN, int PASSES, int EPI, int CS, int EW = 8>
int query_max_clusters(int num_sms) {
  int n = num_sms / (CG * CS);
  if (CG * CS > 2) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(static_cast<unsigned>(num_sms / (CG * CS) * (CG * CS)));
    cfg.blockDim = dim3(Cfg<CG, BN, PASSES, EW>::kThreads);
    cfg.dynamicSmemBytes = Cfg<CG, BN, PASSES, EW>::kSmemBytes;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG * CS;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int q = 0;
    if (cudaOccupancyMaxActiveClusters(&q, gemm_tc_kernel<CG, BN, PASSES, EPI, CS, EW>, &cfg) == cudaSuccess && q > 0 && q < n)
      n = q;
    (void)cudaGetLastError();
  }
  return n;
}

// Asked once per kernel instance.  A function-local static is initialised exactly once even when handles are created
// from several threads at the same time (C++11 thread-safe initialisation).
template <int CG, int BN, int PASSES, int EPI, int CS, int EW = 8>
int max_clusters(int num_sms) {
  static const int cached = query_max_clusters<CG, BN, PASSES, EPI, CS, EW>(num_sms);
  return cached;
}

template <int CG, int BN, int PASSES, int EPI, int CS = 1, int EW = 8>
cudaError_t launch_one(const GemmMaps& m, const GemmParams& p, int num_sms, cudaStream_t st) {
  using C = Cfg<CG, BN, PASSES, EW>;
  auto kern = gemm_tc_kernel<CG, BN, PASSES, EPI, CS, EW>;
  const int tiles_m = (p.M + BM * CG - 1) / (BM * CG);
  const int n_tiles = ((tiles_m + CS - 1) / CS) * (p.N / BN);
  const int max_units = max_clusters<CG, BN, PASSES, EPI, CS, EW>(num_sms);
  const int units = n_tiles < max_units ? n_tiles : max_units;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(static_cast<unsigned>(units * CG * CS));
  cfg.blockDim = dim3(C::kThreads);
  cfg.dynamicSmemBytes = C::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG * CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, m.a_hi, m.a_lo, CS == 2 ? m.b_hi64 : m.b_hi, CS == 2 ? m.b_lo64 : m.b_lo,
                            PASSES == 4 ? m.a_sf : m.a_hi, PASSES == 4 ? m.b_sf : m.b_hi, EPI == EPI_F32_RED ? m.out : m.a_hi, p);
}

template <int CG, int BN, int PASSES, int EPI, int CS = 1, int EW = 8>
cudaError_t configure_one() {
  return cudaFuncSetAttribute(gemm_tc_kernel<CG, BN, PASSES, EPI, CS, EW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              Cfg<CG, BN, PASSES, EW>::kSmemBytes);
}

}  // namespace

#define D3D_FOR_ALL_GEMMS(X)                                                                        \
  X(1, 128, 3, EPI_F32) X(1, 128, 3, EPI_GELU_SPLIT) X(1, 128, 3, EPI_QKV16)                         \
  X(1, 256, 3, EPI_F32) X(1, 256, 3, EPI_GELU_SPLIT) X(1, 256, 3, EPI_QKV16)                         \
  X(1, 128, 1, EPI_F32) X(1, 128, 1, EPI_GELU_SPLIT) X(1, 128, 1, EPI_QKV16)                         \
  X(1, 256, 1, EPI_F32) X(1, 256, 1, EPI_GELU_SPLIT) X(1, 256, 1, EPI_QKV16)                         \
  X(2, 256, 3, EPI_F32) X(2, 256, 3, EPI_GELU_SPLIT) X(2, 256, 3, EPI_QKV16)                         \
  X(2, 256, 1, EPI_F32) X(2, 256, 1, EPI_GELU_SPLIT) X(2, 256, 1, EPI_QKV16)                         \
  X(1, 256, 2, EPI_F32) X(1, 256, 2, EPI_GELU_SPLIT) X(1, 256, 2, EPI_QKV16)                         \
  X(2, 256, 2, EPI_F32) X(2, 256, 2, EPI_GELU_SPLIT) X(2, 256, 2, EPI_QKV16)

// Opt in to >48 KiB dynamic shared memory for every instantiation (once per device, outside graph capture).
cudaError_t configure_gemm_tc() {
  cudaError_t e;
#define D3D_CFG(CG_, BN_, PASSES_, EPI_) \
  if ((e = configure_one<CG_, BN_, PASSES_, EPI_>()) != cudaSuccess) return e;
  D3D_FOR_ALL_GEMMS(D3D_CFG)
#undef D3D_CFG
  if ((e = configure_one<2, 256, 2, EPI_F32, 2>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 2, EPI_GELU_SPLIT, 2>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 2, EPI_QKV16, 2>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 2, EPI_GELU_SPLIT, 1, 16>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 2, EPI_QKV16, 1, 16>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 2, EPI_F32_LN>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 2, EPI_F32, 1, 16>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 4, EPI_F32>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 4, EPI_GELU_SPLIT>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 4, EPI_QKV16>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 4, EPI_F32, 1, 16>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 4, EPI_GELU_SPLIT, 1, 16>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 4, EPI_QKV16, 1, 16>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 4, EPI_F32_RED>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 4, EPI_F32_EMIT>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 4, EPI_F32_EMIT, 1, 16>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 4, EPI_GELU_DLN>()) != cudaSuccess) return e;
  if ((e = configure_one<2, 256, 4, EPI_GELU_DLN, 1, 16>()) != cudaSuccess) return e;
  return cudaSuccess;
}

cudaError_t launch_gemm_tc(const GemmMaps& maps, const GemmParams& p, int epi, int passes, int bn, int cta_group,
                           int pair_cluster, int epi_warps, int num_sms, cudaStream_t st) {
  if (p.M <= 0) return cudaSuccess;
  if (passes == 4) {
    // FMT_F4C: CTA-pair 256 x 256 tiles only; K in whole e2m1 stages (256 nibbles = 128 bytes of the K-byte c4 row)
    if (p.N % 256 != 0 || p.K % 128 != 0 || epi == EPI_F32_LN) return cudaErrorInvalidValue;
    if (epi == EPI_QKV16 && p.N != 3 * kC) return cudaErrorInvalidValue;
    if ((epi == EPI_GELU_SPLIT || epi == EPI_GELU_DLN) && (!p.out_sf || p.N > 1024)) return cudaErrorInvalidValue;
    // deferred LayerNorm: statistics parts of 64 columns, eight per 512-wide row
    if (epi == EPI_F32_EMIT && (p.N != kC || !p.residual || !p.emit_hi || !p.emit_c4 || !p.emit_sf || !p.ln_stats))
      return cudaErrorInvalidValue;
    if (epi == EPI_GELU_DLN && (p.K != kC || !p.ln_stats || !p.ln_colsum)) return cudaErrorInvalidValue;
    if (epi == EPI_F32_RED && (!p.out_f32 || epi_warps == 16)) return cudaErrorInvalidValue;
    if (epi_warps == 16) {
      if (epi == EPI_F32) return launch_one<2, 256, 4, EPI_F32, 1, 16>(maps, p, num_sms, st);
      if (epi == EPI_GELU_SPLIT) return launch_one<2, 256, 4, EPI_GELU_SPLIT, 1, 16>(maps, p, num_sms, st);
      if (epi == EPI_F32_EMIT) return launch_one<2, 256, 4, EPI_F32_EMIT, 1, 16>(maps, p, num_sms, st);
      if (epi == EPI_GELU_DLN) return launch_one<2, 256, 4, EPI_GELU_DLN, 1, 16>(maps, p, num_sms, st);
      return launch_one<2, 256, 4, EPI_QKV16, 1, 16>(maps, p, num_sms, st);
    }
    if (epi == EPI_F32) return launch_one<2, 256, 4, EPI_F32>(maps, p, num_sms, st);
    if (epi == EPI_F32_RED) return launch_one<2, 256, 4, EPI_F32_RED>(maps, p, num_sms, st);
    if (epi == EPI_GELU_SPLIT) return launch_one<2, 256, 4, EPI_GELU_SPLIT>(maps, p, num_sms, st);
    if (epi == EPI_F32_EMIT) return launch_one<2, 256, 4, EPI_F32_EMIT>(maps, p, num_sms, st);
    if (epi == EPI_GELU_DLN) return launch_one<2, 256, 4, EPI_GELU_DLN>(maps, p, num_sms, st);
    return launch_one<2, 256, 4, EPI_QKV16>(maps, p, num_sms, st);
  }
  if (epi == EPI_F32_EMIT || epi == EPI_GELU_DLN || epi == EPI_F32_RED) return cudaErrorInvalidValue;     // FMT_F4C kernel only
  if (cta_group == 2 || passes == 2) bn = 256;
  if (epi == EPI_F32_LN) {
    // needs: both 256-column halves of a row tile on the same CTA pair, back to back, in accumulators 0 and 1
    if (cta_group != 2 || passes != 2 || p.N != 2 * 256 || !p.n_inner || !p.residual || !p.ln_gamma || !p.ln_beta ||
        !p.ln_hi || !p.ln_second)
      return cudaErrorInvalidValue;
    return launch_one<2, 256, 2, EPI_F32_LN>(maps, p, num_sms, st);
  }
  if (epi_warps == 16 && cta_group == 2 && passes == 2 && pair_cluster != 2) {
    if (epi == EPI_F32) return launch_one<2, 256, 2, EPI_F32, 1, 16>(maps, p, num_sms, st);
    if (epi == EPI_GELU_SPLIT) return launch_one<2, 256, 2, EPI_GELU_SPLIT, 1, 16>(maps, p, num_sms, st);
    if (epi == EPI_QKV16) return launch_one<2, 256, 2, EPI_QKV16, 1, 16>(maps, p, num_sms, st);
  }
  if (p.K % BK != 0 || p.N % bn != 0 || (bn != 128 && bn != 256)) return cudaErrorInvalidValue;
  if (epi == EPI_QKV16 && p.N != 3 * kC) return cudaErrorInvalidValue;
  if (pair_cluster == 2 && cta_group == 2 && passes == 2) {
    if (epi == EPI_F32) return launch_one<2, 256, 2, EPI_F32, 2>(maps, p, num_sms, st);
    if (epi == EPI_GELU_SPLIT) return launch_one<2, 256, 2, EPI_GELU_SPLIT, 2>(maps, p, num_sms, st);
    return launch_one<2, 256, 2, EPI_QKV16, 2>(maps, p, num_sms, st);
  }
#define D3D_DISPATCH(CG_, BN_, PASSES_, EPI_)                                   \
  if (cta_group == CG_ && bn == BN_ && passes == PASSES_ && epi == EPI_)        \
    return launch_one<CG_, BN_, PASSES_, EPI_>(maps, p, num_sms, st);
  D3D_FOR_ALL_GEMMS(D3D_DISPATCH)
#undef D3D_DISPATCH
  return cudaErrorInvalidValue;
}

// ---------------------------------------------------------------------------------------------------
// Tensor-map construction (driver entry point fetched through the runtime: no link-time libcuda dependency)
// ---------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// D3D_TMA_L2_PROMO: L2 promotion of the GEMM's tensor maps (0 none, 1 64 B, 2 128 B, 3 256 B; read when a map is encoded)
static CUtensorMapL2promotion l2_promotion() {
  const char* v = getenv("D3D_TMA_L2_PROMO");
  const int k = (v && *v) ? atoi(v) : 3;
  return k == 0 ? CU_TENSOR_MAP_L2_PROMOTION_NONE : k == 1 ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B
       : k == 2 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B : CU_TENSOR_MAP_L2_PROMOTION_L2_256B;
}

static EncodeTiledFn query_encode_tiled() {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  return (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) ? reinterpret_cast<EncodeTiledFn>(fn) : nullptr;
}

// The driver's cuTensorMapEncodeTiled, fetched once (thread-safe initialisation of a function-local static).
static EncodeTiledFn encode_tiled() {
  static const EncodeTiledFn fn = query_encode_tiled();
  return fn;
}

int make_operand_map(CUtensorMap* out, const __half* base, int64_t rows, int64_t K, int box_rows) {
  const EncodeTiledFn encode = encode_tiled();
  if (!encode) return -1;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(K) * 2};
  cuuint32_t box[2] = {BK, static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(base), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, l2_promotion(),
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : -static_cast<int>(r) - 1000;
}


// uint8 [rows, row_bytes] row-major array (the c8 arrays of FMT_F8C): {128 bytes x 128 rows} boxes, SWIZZLE_128B
int make_operand_map_u8(CUtensorMap* out, const void* base, int64_t rows, int64_t row_bytes, int box_rows) {
  const EncodeTiledFn encode = encode_tiled();
  if (!encode) return -1;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(row_bytes), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(row_bytes)};
  cuuint32_t box[2] = {128, static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, l2_promotion(),
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : -static_cast<int>(r) - 1000;
}

int make_f32_tile_map(CUtensorMap* out, const float* base, int64_t rows, int N) {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) return -1;
  EncodeTiledFn encode = reinterpret_cast<EncodeTiledFn>(fn);
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(N), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(N) * 4};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, l2_promotion(),
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : -static_cast<int>(r) - 1000;
}

// FMT_F4C scale-factor array (operand.cuh) viewed as [total_bytes / 256][256] bytes: {256 x 4} boxes, no swizzle, so a
// box lands in shared memory as 1 KB of consecutive bytes = two 512-byte atoms (the two k-atoms of one e2m1 stage)
int make_sf_map(CUtensorMap* out, const void* base, int64_t total_bytes) {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) return -1;
  EncodeTiledFn encode = reinterpret_cast<EncodeTiledFn>(fn);
  if (total_bytes % 1024 != 0) return -2;
  cuuint64_t dims[2] = {256, static_cast<cuuint64_t>(total_bytes / 256)};
  cuuint64_t strides[1] = {256};
  cuuint32_t box[2] = {256, 4};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, l2_promotion(),
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : -static_cast<int>(r) - 1000;
}

}  // namespace d3d
