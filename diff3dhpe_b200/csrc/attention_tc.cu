// G-tattn / G-sattn on the 5th-generation tensor cores: the GRAND attention core (MODEL:76-83) as ONE persistent
// tcgen05 / TMEM / TMA kernel with two modes -- temporal (F > 64 frames per sequence, the rearranges of MODEL:121,133
// folded into the addressing) and spatial (17 joints per frame, 7 frames per 128-row tile with a block-diagonal mask,
// see softmax_row_spatial).  The description below is the temporal mode.
//
//     O = softmax(Q K^T * hd^-0.5) V  -  V[query]            ((P - I) V == P V - V, SURVEY.md K12)
//
// Why not the mma.sync kernel of attention_mma.cu: at F = 243 it is bound by shared-memory bandwidth (every warp
// re-reads all of K and V through ldmatrix for each 16-query tile) and by issue slots (fragment shuffles, online-
// softmax rescaling): 9.3 ms per call at cfg3 against an HBM floor of 2 ms (profiles/r01h_bench.json).  Here
//   * one work unit = (clip b, joint j, head h); its Q, K, V_hi slabs ({F rows x 128 B}, row stride J tokens) are
//     gathered by 4-D TMA boxes straight into the canonical K-major SWIZZLE_128B layout (rows >= F are zero-filled
//     by the TMA unit), no transposed copy of the activations exists;
//   * S = Q K^T is ONE tcgen05.mma chain per 128-query tile (M = 128, N = F rounded up to 16, K = 64) into TMEM;
//   * each of 128 threads owns one query ROW of S (tcgen05.ld, lane = row): the softmax needs no shuffles, no
//     online rescaling (two passes over TMEM: max, then exp2 / sum), and writes P as packed fp16 back into the
//     same TMEM columns (tcgen05.st) -- P never touches shared memory;
//   * O = P V is a second tcgen05.mma chain with A = P from TMEM and B = V from shared memory as an MN-major
//     operand (V rows are keys, the contraction index), accumulating into the (dead) upper half of S;
//   * the epilogue normalises, subtracts the exact V row (v_hi from shared memory + v_lo, which a TMA load drops into
//     the Q tile once S is complete), packs the GEMM A-operand format in place and leaves through TMA stores (rows
//     >= F are clipped by the hardware).
// One CTA per SM keeps two 128-query tiles ("slots", 256 TMEM columns each) and two or four units (shared-memory
// stages) in flight: while one slot runs its softmax on the CUDA cores the other is in its tensor-core phase, and the next
// unit's Q/K/V are already landing.  Measured history and ncu evidence: DESIGN.md section 4.2.
//
// Warp roles (384 threads): 0..3 softmax + epilogue of slot 0 (TMEM lane quadrant = warp & 3), 4..7 of slot 1,
// 8 = TMA producer, 9 = MMA issuer and TMEM allocator, 10..11 idle (they complete the control warpgroup).
#include <cstdlib>
#include "kernels.cuh"
#include "operand.cuh"
// The barrier waits of this kernel sit on a per-item latency chain (MMA -> softmax -> MMA -> epilogue): the sleeping
// wait of ptx.cuh costs +4 % here (wake-up latency; profiles/r01zd_bench_*.json: 489 -> 501 ms per cfg3 step for both
// modes) while it gains 0.5 % in the GEMM, whose waits have slack.  Busy try_wait polling in this file.
#define D3D_MBAR_SUSPEND_NS 0
#include "ptx.cuh"

namespace d3d {
namespace {

constexpr int kTcThreads = 384;           // 3 warpgroups: softmax slot 0, softmax slot 1, control (TMA, MMA, 2 idle warps)
// 384 threads launch with 168 registers each (3 warps per SM sub-partition x 168 x 32 <= 16 384).  The softmax rows
// keep four 32-column TMEM batches in flight (128 registers): the control warpgroup hands its surplus over with
// setmaxnreg (2 x 128 x (216 - 168) <= 128 x (168 - 40)); each setmaxnreg sits inside its role branch so that ptxas
// allocates per branch.
constexpr int kCtrlRegs = 40, kSoftmaxRegs = 216;
static_assert(2 * 128 * (kSoftmaxRegs - 168) <= 128 * (168 - kCtrlRegs), "setmaxnreg pool overdrawn");
constexpr int kSpatialRows = 7 * 17;      // spatial mode: tokens (7 frames) per unit
constexpr int kTile = 128 * 128;          // bytes of one {64 halves x 128 rows} box
constexpr int kSlotCols = 256;            // TMEM columns of one slot: S up to 256 fp32; P aliases [0,128), O [128,192)
constexpr int kOCol = 128;
constexpr float kScaleLog2e = 0.125f * 1.4426950408889634f;   // head_dim ** -0.5 (MODEL:65) in the exp2 domain

// NSLOT = 128-query tiles in flight per CTA (each with its own 4 softmax warps and 256 TMEM columns).  Shipped: 2.  (A first version with one slot and two CTAs per SM measured 430 ms
// per cfg3 step against 398 ms, profiles/r01m_bench_slots*.json.)
constexpr int kMaxStages = 4;
template <int NSLOT>
struct TcBars {
  uint64_t full[kMaxStages];        // TMA bytes of the unit in this stage landed          (producer -> MMA)
  uint64_t stage_free[kMaxStages];  // every tile of the unit has left this stage           (epilogues -> producer)
  uint64_t s_full[NSLOT];       // S = Q K^T complete in this slot's TMEM columns           (MMA -> softmax)
  uint64_t p_full[NSLOT];       // P written to TMEM by all 128 rows                        (softmax -> MMA)
  uint64_t o_full[NSLOT];       // O = P V complete                                         (MMA -> epilogue)
  uint64_t tmem_free[NSLOT];    // O read out: the columns may receive the next S           (epilogue -> MMA)
  uint64_t vlo_full[NSLOT];     // v_lo rows of the tile landed in the (dead) Q tile        (TMA -> epilogue)
  uint64_t staged[NSLOT];       // the tile's output rows are staged in shared memory       (epilogue -> store warp)
  uint64_t stg_free[NSLOT];     // the TMA stores have read the slot's staging buffer       (store warp -> epilogue)
  uint32_t tmem_base;
};

// D3D_ATTN_STORE_WARP = 1: the TMA stores of a tile and the wait for them to have read shared memory are issued by an
// otherwise idle warp of the control warpgroup (one per slot) instead of by row 0 of the slot's softmax warps, whose warp
// would sit in cp.async.bulk.wait_group.read while the next S of the slot is already complete (the slot's four warps
// arrive on p_full together, so the wait was on every tile's critical path).
#ifndef D3D_ATTN_STORE_WARP
#define D3D_ATTN_STORE_WARP 1
#endif

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {      // one cvt.rn.f16x2.f32
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// MN-major SWIZZLE_128B operand (V as B of P.V: rows = keys = contraction index, 64 head channels contiguous):
// canonical layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units -> 8 keys x 128 B per swizzle atom, next 8 keys
// SBO = 1024 B further; one atom wide in N (64 halves), so LBO is unused.
__device__ __forceinline__ uint64_t make_desc_mn_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3ffffu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}


__device__ __forceinline__ float row_sum(const ptx::f32x2 (&ls)[2]) {
  float a, b, c, d;
  ptx::unpack2(ls[0], a, b);
  ptx::unpack2(ls[1], c, d);
  return (a + b) + (c + d);
}

// One query row (= this thread's TMEM lane) of S -> P, two passes over tensor memory:
//   pass 1: m = max over the F real keys;   pass 2: P = exp2(S c - m c) as packed fp16 into columns [0, n/2) of the
//   same slot (column k/2 is written after S columns <= k+1 were read), row sum in fp32.  Returns 1 / sum.
// TMEM reads are issued one batch (two 32-column chunks) ahead of the batch being processed.  NCH > 0: the number of
// chunks is a compile-time constant and F > 32 (NCH - 1), so every offset is an immediate and only the last chunk is
// masked; NCH == 0: runtime chunk count (<= 8).
template <int NCH>
__device__ __forceinline__ float softmax_row(uint32_t taddr, int F, int n_chunks_rt) {
  constexpr int kMax = NCH > 0 ? NCH : 8;
  const int n = NCH > 0 ? NCH : n_chunks_rt;
  uint32_t a0[32], a1[32], b0[32], b1[32];
  float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
  auto full = [&](int c) { return (NCH > 0 && c < NCH - 1) || (c + 1) * 32 <= F; };
  auto max_chunk = [&](const uint32_t (&rr)[32], int c) {
    if (full(c)) {
#pragma unroll
      for (int e = 0; e < 32; ++e) mx[e & 3] = fmaxf(mx[e & 3], __uint_as_float(rr[e]));
    } else {
#pragma unroll
      for (int e = 0; e < 32; ++e)
        if (c * 32 + e < F) mx[e & 3] = fmaxf(mx[e & 3], __uint_as_float(rr[e]));
    }
  };
  ptx::tmem_ld_32x32(taddr, a0);
  if (1 < n) ptx::tmem_ld_32x32(taddr + 32, a1);
#pragma unroll
  for (int c = 0; c < kMax; c += 4) {
    if (c < n) {
      ptx::tmem_ld_wait();
      if (c + 2 < n) ptx::tmem_ld_32x32(taddr + (c + 2) * 32, b0);
      if (c + 3 < n) ptx::tmem_ld_32x32(taddr + (c + 3) * 32, b1);
      max_chunk(a0, c);
      if (c + 1 < n) max_chunk(a1, c + 1);
    }
    if (c + 2 < n) {
      ptx::tmem_ld_wait();
      if (c + 4 < n) ptx::tmem_ld_32x32(taddr + (c + 4) * 32, a0);
      if (c + 5 < n) ptx::tmem_ld_32x32(taddr + (c + 5) * 32, a1);
      max_chunk(b0, c + 2);
      if (c + 3 < n) max_chunk(b1, c + 3);
    }
  }
  // pass 2 starts streaming before the max is reduced
  ptx::tmem_ld_32x32(taddr, a0);
  if (1 < n) ptx::tmem_ld_32x32(taddr + 32, a1);
  const float nmxs = -fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3])) * kScaleLog2e;
  // packed pairs (FFMA2 / FADD2): the scale-and-shift and the row sum cost one fma-pipe slot per TWO keys
  ptx::f32x2 ls[2] = {ptx::splat2(0.f), ptx::splat2(0.f)};
  const ptx::f32x2 sc2 = ptx::splat2(kScaleLog2e), nm2 = ptx::splat2(nmxs);
  auto exp_chunk = [&](const uint32_t (&rr)[32], int c) {
    uint32_t pk[16];
    const bool whole = full(c);
#pragma unroll
    for (int e = 0; e < 16; ++e) {
      float t0, t1;
      ptx::unpack2(ptx::fma2(ptx::pack2(__uint_as_float(rr[2 * e]), __uint_as_float(rr[2 * e + 1])), sc2, nm2), t0, t1);
      const int col = c * 32 + 2 * e;
      const float e0 = (whole || col < F) ? ex2_approx(t0) : 0.f;
      const float e1 = (whole || col + 1 < F) ? ex2_approx(t1) : 0.f;
      ls[e & 1] = ptx::add2(ls[e & 1], ptx::pack2(e0, e1));
      pk[e] = pack_f16x2(e0, e1);
    }
    ptx::tmem_st_32x16(taddr + c * 16, pk);
  };
#pragma unroll
  for (int c = 0; c < kMax; c += 4) {
    if (c < n) {
      ptx::tmem_ld_wait();
      if (c + 2 < n) ptx::tmem_ld_32x32(taddr + (c + 2) * 32, b0);
      if (c + 3 < n) ptx::tmem_ld_32x32(taddr + (c + 3) * 32, b1);
      exp_chunk(a0, c);
      if (c + 1 < n) exp_chunk(a1, c + 1);
    }
    if (c + 2 < n) {
      ptx::tmem_ld_wait();
      if (c + 4 < n) ptx::tmem_ld_32x32(taddr + (c + 4) * 32, a0);
      if (c + 5 < n) ptx::tmem_ld_32x32(taddr + (c + 5) * 32, a1);
      exp_chunk(b0, c + 2);
      if (c + 3 < n) exp_chunk(b1, c + 3);
    }
  }
  ptx::tmem_st_wait();
  return rcp_approx(row_sum(ls));
}

// Spatial mode: the 128-row tile holds 7 frames x 17 joints (rows 119..127 belong to the next unit and are never
// stored); query row r attends only the 17 keys of its own frame, columns [17 (r / 17), +17) of S.  A warp's 32 rows
// touch at most 3 frames, i.e. a 51-column window inside the three aligned 32-column chunks starting at chunk
// CS = wq >> 1 (wq = TMEM lane quadrant).  P is written for all 128 keys (zero outside the window), so the P.V chain
// is the same as in the temporal mode.
//
// spatial_window<CS, FR>: the 17 keys of frame FR with COMPILE-TIME register indices -- no per-column masks or selects
// (the masked form over all 96 loaded columns cost ~7 instructions per column, 665 per row; this one ~70 per frame, and
// a warp runs at most three of them divergently).  Writes the packed fp16 P pairs of its window into pk (zero elsewhere)
// and returns the row sum.
template <int CS, int FR>
__device__ __forceinline__ float spatial_window(const uint32_t (&a)[32], const uint32_t (&b)[32], const uint32_t (&c)[32],
                                                uint32_t (&pk0)[16], uint32_t (&pk1)[16], uint32_t (&pk2)[16]) {
  constexpr int L = 17 * FR - 32 * CS;          // first window column among the 96 loaded ones
  static_assert(L >= 0 && L + 17 <= 96, "frame window outside the loaded chunks");
  float sv[18];
#pragma unroll
  for (int k = 0; k < 17; ++k) {
    const int li = L + k;
    sv[k] = __uint_as_float(li < 32 ? a[li & 31] : li < 64 ? b[li & 31] : c[li & 31]);
  }
  sv[17] = sv[16];                              // pads the last pair; never stored or summed
  float mx = sv[0];
#pragma unroll
  for (int k = 1; k < 17; k += 2) mx = fmaxf(mx, fmaxf(sv[k], sv[k + 1]));
  const ptx::f32x2 sc2 = ptx::splat2(kScaleLog2e), nm2 = ptx::splat2(-mx * kScaleLog2e);
  float ev[18];
  ptx::f32x2 ls = ptx::splat2(0.f);
#pragma unroll
  for (int k = 0; k < 18; k += 2) {
    float t0, t1;
    ptx::unpack2(ptx::fma2(ptx::pack2(sv[k], sv[k + 1]), sc2, nm2), t0, t1);
    ev[k] = ex2_approx(t0);
    ev[k + 1] = k + 1 < 17 ? ex2_approx(t1) : 0.f;
    ls = ptx::add2(ls, ptx::pack2(ev[k], ev[k + 1]));
  }
#pragma unroll
  for (int pi = L / 2; pi <= (L + 16) / 2; ++pi) {
    const int k0 = 2 * pi - L, k1 = k0 + 1;
    const uint32_t v = pack_f16x2(k0 >= 0 && k0 < 17 ? ev[k0 < 0 ? 0 : k0] : 0.f, k1 >= 0 && k1 < 17 ? ev[k1] : 0.f);
    if (pi < 16) pk0[pi & 15] = v;
    else if (pi < 32) pk1[pi & 15] = v;
    else pk2[pi & 15] = v;
  }
  float s0, s1;
  ptx::unpack2(ls, s0, s1);
  return s0 + s1;
}

__device__ __forceinline__ float softmax_row_spatial(uint32_t taddr, int row_l, int wq) {
  const int cs = wq >> 1;
  uint32_t a[32], b[32], c[32];
  ptx::tmem_ld_32x32(taddr + cs * 32, a);
  ptx::tmem_ld_32x32(taddr + cs * 32 + 32, b);
  ptx::tmem_ld_32x32(taddr + cs * 32 + 64, c);
  uint32_t pk0[16], pk1[16], pk2[16], z[16];
#pragma unroll
  for (int e = 0; e < 16; ++e) pk0[e] = pk1[e] = pk2[e] = z[e] = 0u;
  ptx::tmem_ld_wait();
  const int fr = row_l < 119 ? row_l / 17 : 6;    // rows 119..127 (next unit's tokens, never stored) ride along with frame 6
  float sum;
  if (cs == 0) {
    switch (fr) {
      case 0: sum = spatial_window<0, 0>(a, b, c, pk0, pk1, pk2); break;
      case 1: sum = spatial_window<0, 1>(a, b, c, pk0, pk1, pk2); break;
      case 2: sum = spatial_window<0, 2>(a, b, c, pk0, pk1, pk2); break;
      default: sum = spatial_window<0, 3>(a, b, c, pk0, pk1, pk2); break;
    }
  } else {
    switch (fr) {
      case 3: sum = spatial_window<1, 3>(a, b, c, pk0, pk1, pk2); break;
      case 4: sum = spatial_window<1, 4>(a, b, c, pk0, pk1, pk2); break;
      case 5: sum = spatial_window<1, 5>(a, b, c, pk0, pk1, pk2); break;
      default: sum = spatial_window<1, 6>(a, b, c, pk0, pk1, pk2); break;
    }
  }
  __syncwarp();                                   // tcgen05.st is .sync.aligned: the frames of the warp reconverge here
  ptx::tmem_st_32x16(taddr + cs * 16, pk0);
  ptx::tmem_st_32x16(taddr + cs * 16 + 16, pk1);
  ptx::tmem_st_32x16(taddr + cs * 16 + 32, pk2);
  ptx::tmem_st_32x16(taddr + (cs == 0 ? 48 : 0), z);      // the 32 keys this warp did not load
  ptx::tmem_st_wait();
  return rcp_approx(sum);
}

// Packed temporal mode (F <= 64; cfg4's F = 27): G = 4 (F <= 32) or 2 sequences -- the same (clip, head) of G consecutive
// joints -- share one 128-row tile, row r = f G + jj (the {64 channels, G joints, 128 / G frames} TMA box lands exactly so).
// Query row r attends the keys of its own joint only: columns c with c % G == r % G and c / G < F.  One pass over the
// 128 columns for the max, one for exp2 / sum; P is zero elsewhere, so the P.V chain is the same as in the other modes.
__device__ __forceinline__ float softmax_row_packed(uint32_t taddr, int F, int G, int row_l) {
  const int jj = row_l & (G - 1);
  const uint32_t vm = (G == 4 ? 0x11111111u : 0x55555555u) << jj;      // own-joint columns of any aligned 32-column chunk
  const int nk = F * G;                                                // columns >= nk are frames >= F (zero-filled rows)
  uint32_t sv[4][32];
#pragma unroll
  for (int c = 0; c < 4; ++c) ptx::tmem_ld_32x32(taddr + c * 32, sv[c]);
  ptx::tmem_ld_wait();
  float mx = -INFINITY;
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int e = 0; e < 32; ++e)
      if (((vm >> e) & 1u) && c * 32 + e < nk) mx = fmaxf(mx, __uint_as_float(sv[c][e]));
  const ptx::f32x2 sc2 = ptx::splat2(kScaleLog2e), nm2 = ptx::splat2(-mx * kScaleLog2e);
  ptx::f32x2 ls = ptx::splat2(0.f);
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint32_t pk[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) {
      float t0, t1;
      ptx::unpack2(ptx::fma2(ptx::pack2(__uint_as_float(sv[c][2 * e]), __uint_as_float(sv[c][2 * e + 1])), sc2, nm2), t0, t1);
      const int col = c * 32 + 2 * e;
      const float e0 = (((vm >> (2 * e)) & 1u) && col < nk) ? ex2_approx(t0) : 0.f;
      const float e1 = (((vm >> (2 * e + 1)) & 1u) && col + 1 < nk) ? ex2_approx(t1) : 0.f;
      ls = ptx::add2(ls, ptx::pack2(e0, e1));
      pk[e] = pack_f16x2(e0, e1);
    }
    ptx::tmem_st_32x16(taddr + c * 16, pk);
  }
  ptx::tmem_st_wait();
  float s0, s1;
  ptx::unpack2(ls, s0, s1);
  return rcp_approx(s0 + s1);
}

// Work items of a CTA, in order: w = 0, 1, 2, ... ; unit n = w / n_mt (the CTA's n-th unit), 128-query tile
// m = w % n_mt; slot = w % NSLOT (i-th item of that slot, i = w / NSLOT); shared-memory stage = n % n_stage (k-th use,
// k = n / n_stage).  n_stage = 2 when a unit has two tiles (96 KB per unit), 4 when it has one (48 KB): units are
// then loaded two to three items ahead of the tile being processed -- with only two stages the single-tile modes
// (spatial, F <= 128) were bound by the load -> MMA -> softmax -> MMA -> store latency chain of two units in flight
// (ncu: 62 % of the stall samples were softmax warps waiting on s_full / o_full, profiles/r01o_full_attn_tc.md).
// SPATIAL: unit = (clip, group g of 7 frames = 119 consecutive tokens, head); groups never straddle clips (the last
// group of a clip holds F % 7 frames), so a frame's position inside the tile -- and with it every rounding -- depends
// only on its index inside the clip: results are bit-identical under any batch split.  The maps are 2-D token-major
// views encoded with rank 4 (coordinates (channel, token, 0, 0)); n_mt == 1, NKp == 128; the store maps have 119-row
// boxes, the *_tail maps (F % 7) * 17-row boxes.  J carries the groups per clip.
// PACKED: G = `pk_g` joints per tile (softmax_row_packed); J then counts the joint GROUPS per clip and `j_tok` the joints.
template <int FMT, int NSLOT, int NCH, bool SPATIAL, bool PACKED = false>
__global__ void __launch_bounds__((4 * NSLOT + 4) * 32, 1)
attn_temporal_tc_kernel(const __grid_constant__ CUtensorMap tm_qkv, const __grid_constant__ CUtensorMap tm_hi,
                        const __grid_constant__ CUtensorMap tm_second, const __grid_constant__ CUtensorMap tm_hi_tail,
                        const __grid_constant__ CUtensorMap tm_second_tail, uint8_t* __restrict__ sf_out, int F, int J,
                        int n_units, int n_mt, int NKp, int n_stage, int pk_g = 1, int j_tok = 0) {
  static_assert(!PACKED || (!SPATIAL && NCH == 0), "the packed mode is a temporal mode with a runtime chunk count");
  // NSLOT == 3 (single-tile modes, S only 128 columns wide, FMT_F4C): three 128-column slots, three softmax warpgroups
  // (512 threads, 128 registers at launch, control 40 / softmax 152), P aliases [0, 64), O [64, 128), 8 KB of staging per slot
  static_assert(NSLOT == 2 || (NSLOT == 3 && FMT == FMT_F4C && (SPATIAL || PACKED)), "three slots: single-tile F4C modes only");
  constexpr int kSC = NSLOT == 2 ? kSlotCols : 128;            // TMEM columns per slot
  constexpr int kOC = NSLOT == 2 ? kOCol : 64;                 // O accumulator inside the slot
  constexpr int kStgSlot = NSLOT == 2 ? kTile : 8192;          // staging bytes per slot
  constexpr int kTmemCols = NSLOT == 2 ? 512 : 512;            // power of two >= NSLOT * kSC
  constexpr int kSmxRegs = NSLOT == 2 ? kSoftmaxRegs : 152;
  static_assert(NSLOT != 3 || 3 * 128 * (152 - 128) <= 128 * (128 - kCtrlRegs), "setmaxnreg pool overdrawn");
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int stage_bytes = 3 * n_mt * kTile;          // Q tiles | K tiles | V tiles of one unit
  uint8_t* StgAll = smem + n_stage * stage_bytes;    // 16 KB per slot: second-part staging of one 128-row output tile
  TcBars<NSLOT>* bars = reinterpret_cast<TcBars<NSLOT>*>(StgAll + NSLOT * kStgSlot);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int kTmaWarp = 4 * NSLOT, kMmaWarp = 4 * NSLOT + 1;
  const int n_local = blockIdx.x < n_units ? (n_units - 1 - static_cast<int>(blockIdx.x)) / static_cast<int>(gridDim.x) + 1 : 0;
  const int W = n_local * n_mt;

  if (warp == kTmaWarp && ptx::elect_one()) {
    ptx::prefetch_tensormap(&tm_qkv);
    ptx::prefetch_tensormap(&tm_hi);
    ptx::prefetch_tensormap(&tm_second);
    for (int s = 0; s < n_stage; ++s) {
      ptx::mbar_init(&bars->full[s], 1);
      ptx::mbar_init(&bars->stage_free[s], n_mt);
    }
#pragma unroll
    for (int s = 0; s < NSLOT; ++s) {
      ptx::mbar_init(&bars->s_full[s], 1);
      ptx::mbar_init(&bars->p_full[s], 128);
      ptx::mbar_init(&bars->o_full[s], 1);
      ptx::mbar_init(&bars->tmem_free[s], 128);
      ptx::mbar_init(&bars->vlo_full[s], 1);
      ptx::mbar_init(&bars->staged[s], 1);
      ptx::mbar_init(&bars->stg_free[s], 1);
    }
    ptx::fence_barrier_init();
  }
  if (warp == kMmaWarp) ptx::tmem_alloc<kTmemCols>(&bars->tmem_base);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  if (warp == kTmaWarp) {
    // ------------------------------------------------------------------ TMA producer
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kCtrlRegs));
    if (ptx::elect_one()) {
      for (int n = 0; n < n_local; ++n) {
        const int unit = blockIdx.x + n * gridDim.x;
        const int seq = unit >> 3, h = unit & 7;
        int b = seq / J, j = seq - b * J;
        if (SPATIAL) { j = (b * F + 7 * j) * 17; b = 0; }        // token coordinate of the group's first row
        if (PACKED) j *= pk_g;                                   // first joint of the group
        const int stage = n % n_stage, k = n / n_stage;
        uint8_t* Qs = smem + stage * stage_bytes;
        uint8_t* Ks = Qs + n_mt * kTile;
        uint8_t* Vs = Ks + n_mt * kTile;
        ptx::mbar_wait(&bars->stage_free[stage], (k & 1) ^ 1);
        ptx::mbar_arrive_expect_tx(&bars->full[stage], 3 * n_mt * kTile);
        for (int t = 0; t < n_mt; ++t) {
          ptx::tma_load_4d(Ks + t * kTile, &tm_qkv, &bars->full[stage], kC + h * kHd, j, t * 128, b);
          ptx::tma_load_4d(Qs + t * kTile, &tm_qkv, &bars->full[stage], h * kHd, j, t * 128, b);
          ptx::tma_load_4d(Vs + t * kTile, &tm_qkv, &bars->full[stage], 2 * kC + h * kHd, j, t * 128, b);
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------------------------------------------ MMA issuer
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kCtrlRegs));
    if (ptx::elect_one()) {
      const uint32_t idesc_qk = ptx::make_idesc_f16(128, static_cast<uint32_t>(NKp), 0);
      const uint32_t idesc_pv = ptx::make_idesc_f16(128, kHd, 0) | (1u << 16);      // B (= V) is MN-major
      const uint32_t s0 = ptx::smem_u32(smem);
      const int n_ks = NKp >> 4;
      auto issue_pv = [&](int w) {           // O[128, 64] = P[128, NKp] (TMEM) . V[NKp, 64], 16 keys per MMA
        const int slot = w % NSLOT, i = w / NSLOT, stage = (w / n_mt) % n_stage;
        const uint32_t sV = s0 + stage * stage_bytes + 2 * n_mt * kTile;
        const uint32_t tcol = tmem_base + slot * kSC;
        ptx::mbar_wait(&bars->p_full[slot], i & 1);
        ptx::tc_fence_after();
        for (int ks = 0; ks < n_ks; ++ks)
          ptx::mma_f16_ts(tcol + kOC, tcol + ks * 8, make_desc_mn_sw128(sV + ks * 2048), idesc_pv, ks != 0 ? 1u : 0u);
        ptx::mma_commit(&bars->o_full[slot]);
      };
      for (int w = 0; w < W; ++w) {
        const int n = w / n_mt, m = w - n * n_mt;
        const int slot = w % NSLOT, i = w / NSLOT, stage = n % n_stage;
        const uint32_t sQ = s0 + stage * stage_bytes, sK = sQ + n_mt * kTile;
        if (m == 0) {
          ptx::mbar_wait(&bars->full[stage], (n / n_stage) & 1);
          ptx::tc_fence_after();
        }
        ptx::mbar_wait(&bars->tmem_free[slot], (i & 1) ^ 1);
        ptx::tc_fence_after();
#pragma unroll
        for (int k = 0; k < 4; ++k)            // S[128, NKp] = Q_m[128, 64] . K[NKp, 64]^T, 16 channels per MMA
          ptx::mma_f16_ss(tmem_base + slot * kSC, ptx::make_desc_k_sw128(sQ + m * kTile + k * 32),
                          ptx::make_desc_k_sw128(sK + k * 32), idesc_qk, k != 0 ? 1u : 0u);
        ptx::mma_commit(&bars->s_full[slot]);
        // the P.V of the item NSLOT-1 back: with two slots, S of this item is already being computed while the other
        // slot's softmax finishes
        if (w >= NSLOT - 1) issue_pv(w - (NSLOT - 1));
      }
      for (int w = W - (NSLOT - 1); w < W; ++w)
        if (w >= 0) issue_pv(w);
    }
  } else if (warp > kMmaWarp) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kCtrlRegs));
    // ------------------------------------------------------------------ store warps: one per slot (D3D_ATTN_STORE_WARP)
    const int sidx = warp - (kMmaWarp + 1);          // store warp 0 serves the even slots, store warp 1 the odd ones
    if (D3D_ATTN_STORE_WARP && ptx::elect_one()) {
      for (int w = 0; w < W; ++w) {
        const int slot = w % NSLOT;
        if ((slot & 1) != sidx) continue;
        uint8_t* Stg = StgAll + slot * kStgSlot;
        const int n = w / n_mt, m = w - n * n_mt;
        const int i = w / NSLOT, stage = n % n_stage;
        const int unit = blockIdx.x + n * gridDim.x;
        const int seq = unit >> 3, h = unit & 7;
        int b = seq / J, j = seq - b * J;
        const bool tail = SPATIAL && j == J - 1 && F % 7 != 0;
        if (SPATIAL) { j = (b * F + 7 * j) * 17; b = 0; }
        if (PACKED) j *= pk_g;
        uint8_t* Qs = smem + stage * stage_bytes;
        ptx::mbar_wait(&bars->staged[slot], i & 1);
        const CUtensorMap* mh = tail ? &tm_hi_tail : &tm_hi;
        const CUtensorMap* ms = tail ? &tm_second_tail : &tm_second;
        ptx::tma_store_4d(mh, Qs + m * kTile, h * kHd, j, m * 128, b);
        if (FMT == FMT_F4C) {
          ptx::tma_store_4d(ms, Stg, h * 32, j, m * 128, b);
          ptx::tma_store_4d(ms, Stg + 4096, (kC >> 1) + h * 32, j, m * 128, b);
        } else {
          ptx::tma_store_4d(ms, Stg, h * kHd, j, m * 128, b);
          if (FMT != FMT_SPLIT16) ptx::tma_store_4d(ms, Stg + 8192, kC + h * kHd, j, m * 128, b);
        }
        ptx::bulk_commit();
        ptx::bulk_wait_read_all();           // Stg / Q_m have been read: the tile has left shared memory
        ptx::mbar_arrive(&bars->stage_free[stage]);
        ptx::mbar_arrive(&bars->stg_free[slot]);
      }
      ptx::bulk_wait_all();
    }
  } else {
    // ------------------------------------------------------------------ softmax + epilogue: thread = query row
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kSmxRegs));
    const int slot = warp >> 2;
    const int row_l = (warp & 3) * 32 + lane;                             // row inside the 128-query tile
    const uint32_t taddr = tmem_base + slot * kSC + (static_cast<uint32_t>((warp & 3) * 32) << 16);
    const int n_chunks = (NKp + 31) >> 5;
    if (!SPATIAL && NCH > 0 && (n_chunks != NCH || F <= 32 * (NCH - 1))) __trap();    // launcher / instantiation mismatch
    if ((SPATIAL || PACKED) && (n_mt != 1 || NKp != 128)) __trap();
    const int sw = (row_l & 7) << 4;                                      // swizzle XOR of this row (bytes)
    const bool issuer = row_l == 0;                                       // issues the slot's TMA stores
    uint8_t* Stg = StgAll + slot * kStgSlot;
    for (int w = slot; w < W; w += NSLOT) {
      const int n = w / n_mt, m = w - n * n_mt;
      const int i = w / NSLOT, stage = n % n_stage;
      const int unit = blockIdx.x + n * gridDim.x;
      const int seq = unit >> 3, h = unit & 7;
      int b = seq / J, j = seq - b * J;
      const bool tail = SPATIAL && j == J - 1 && F % 7 != 0;      // last group of a clip: fewer than 7 frames to store
      if (SPATIAL) { j = (b * F + 7 * j) * 17; b = 0; }
      if (PACKED) j *= pk_g;
      uint8_t* Qs = smem + stage * stage_bytes;
      const uint8_t* Vs = Qs + 2 * n_mt * kTile;
      const int r = m * 128 + row_l;
      ptx::mbar_wait(&bars->s_full[slot], i & 1);
      ptx::tc_fence_after();
      if (issuer) {      // Q_m is dead once S is complete: it receives the v_lo rows of the tile (exact "- V" term)
        ptx::mbar_arrive_expect_tx(&bars->vlo_full[slot], kTile);
        ptx::tma_load_4d(Qs + m * kTile, &tm_qkv, &bars->vlo_full[slot], 3 * kC + h * kHd, j, m * 128, b);
      }
      const float inv = SPATIAL ? softmax_row_spatial(taddr, row_l, warp & 3)
                      : PACKED  ? softmax_row_packed(taddr, F, pk_g, row_l)
                                : softmax_row<NCH>(taddr, F, n_chunks);
      ptx::tc_fence_before();
      ptx::mbar_arrive(&bars->p_full[slot]);

      // ---- while the P.V chain runs: this row's exact "- V" term, -(v_hi + v_lo), as 32 packed fp32 pairs (the v_lo row
      // landed in the dead Q tile long ago; ncu had 15 % of the softmax warps' samples idle on o_full and another 10 % on
      // the shared-memory loads below when they sat inside the epilogue loop, profiles/r01p_full_attn_tc.md)
      ptx::mbar_wait(&bars->vlo_full[slot], i & 1);
      uint8_t* hi_row = Qs + m * kTile + row_l * 128;        // v_lo row in, hi row out (same thread, same 16 bytes)
      const uint8_t* v_row = Vs + static_cast<size_t>(r) * 128;
      ptx::f32x2 nv[32];
      {
        uint4 vh[8], vl[8];
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          vh[g] = *reinterpret_cast<const uint4*>(v_row + ((g << 4) ^ sw));
          vl[g] = *reinterpret_cast<const uint4*>(hi_row + ((g << 4) ^ sw));
        }
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const uint32_t vhw[4] = {vh[g].x, vh[g].y, vh[g].z, vh[g].w};
          const uint32_t vlw[4] = {vl[g].x, vl[g].y, vl[g].z, vl[g].w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&vhw[e]));
            const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&vlw[e]));
            float s0, s1;
            ptx::unpack2(ptx::add2(ptx::pack2(a.x, a.y), ptx::pack2(c.x, c.y)), s0, s1);
            nv[4 * g + e] = ptx::pack2(-s0, -s1);
          }
        }
      }

      // ---- O row out of TMEM, then the columns are free for the next S
      ptx::mbar_wait(&bars->o_full[slot], i & 1);
      ptx::tc_fence_after();
      uint32_t o0[32], o1[32];
      ptx::tmem_ld_32x32(taddr + kOC, o0);
      ptx::tmem_ld_32x32(taddr + kOC + 32, o1);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(&bars->tmem_free[slot]);

      // ---- epilogue: out = O / l - (v_hi + v_lo), packed as the proj GEMM's A operand, staged for the TMA stores
      if (D3D_ATTN_STORE_WARP) {             // the previous tile's stores have read the slot's staging buffer
        if (i > 0) ptx::mbar_wait(&bars->stg_free[slot], (i - 1) & 1);
      } else {
        ptx::bar_sync(1 + slot, 128);        // the issuer is past the read-wait of the previous tile's stores: Stg is free
      }
      const ptx::f32x2 inv2 = ptx::splat2(inv);
      if (FMT == FMT_F4C) {
        // block-scaled operand (operand.cuh): the row's 64 channels are two 32-element scale blocks of each part.
        // Pass 1: x = O inv - (v_hi + v_lo) back into the O registers, hi halves into the (dead) Q row, block maxima of
        // x and of x - hi.  Pass 2: P = q4(x), Q = q4(x - hi) as [128 rows][32 B] tiles for the two TMA stores.
        float ax[2] = {0.f, 0.f}, al[2] = {0.f, 0.f};
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          uint32_t hw[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            uint32_t& ra = g < 4 ? o0[8 * g + 2 * e] : o1[8 * (g & 3) + 2 * e];
            uint32_t& rb = g < 4 ? o0[8 * g + 2 * e + 1] : o1[8 * (g & 3) + 2 * e + 1];
            float x0, x1;
            ptx::unpack2(ptx::fma2(ptx::pack2(__uint_as_float(ra), __uint_as_float(rb)), inv2, nv[4 * g + e]), x0, x1);
            const __half2 h01 = __floats2half2_rn(x0, x1);
            const float2 hf = __half22float2(h01);
            hw[e] = *reinterpret_cast<const uint32_t*>(&h01);
            ax[g >> 2] = fmaxf(ax[g >> 2], fmaxf(fabsf(x0), fabsf(x1)));
            al[g >> 2] = fmaxf(al[g >> 2], fmaxf(fabsf(x0 - hf.x), fabsf(x1 - hf.y)));
            ra = __float_as_uint(x0);
            rb = __float_as_uint(x1);
          }
          *reinterpret_cast<uint4*>(hi_row + ((g << 4) ^ sw)) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
        }
        const uint32_t bp0 = op_ue8m0_of(ax[0]), bp1 = op_ue8m0_of(ax[1]), bq0 = op_ue8m0_of(al[0]), bq1 = op_ue8m0_of(al[1]);
        uint32_t pw[8], qw[8];
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const ptx::f32x2 ip = ptx::splat2(op_ue8m0_inv(g < 4 ? bp0 : bp1)), iq = ptx::splat2(op_ue8m0_inv(g < 4 ? bq0 : bq1));
          uint32_t pa = 0, qa = 0;
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float x0 = __uint_as_float(g < 4 ? o0[8 * g + 2 * e] : o1[8 * (g & 3) + 2 * e]);
            const float x1 = __uint_as_float(g < 4 ? o0[8 * g + 2 * e + 1] : o1[8 * (g & 3) + 2 * e + 1]);
            const float2 hf = __half22float2(__floats2half2_rn(x0, x1));
            float a0, a1, l0, l1;
            ptx::unpack2(ptx::mul2(ptx::pack2(x0, x1), ip), a0, a1);
            ptx::unpack2(ptx::mul2(ptx::sub2(ptx::pack2(x0, x1), ptx::pack2(hf.x, hf.y)), iq), l0, l1);
            pa |= op_e2m1x2(a0, a1) << (8 * e);
            qa |= op_e2m1x2(l0, l1) << (8 * e);
          }
          pw[g] = pa; qw[g] = qa;
        }
        {                                                              // [128 rows][32 B] P tile, then the Q tile
          uint4* stp = reinterpret_cast<uint4*>(Stg + row_l * 32);
          stp[0] = make_uint4(pw[0], pw[1], pw[2], pw[3]);
          stp[1] = make_uint4(pw[4], pw[5], pw[6], pw[7]);
          stp[256] = make_uint4(qw[0], qw[1], qw[2], qw[3]);
          stp[257] = make_uint4(qw[4], qw[5], qw[6], qw[7]);
        }
        // the row's four scale bytes: k-blocks (2h, 2h+1) of part P and (16 + 2h, 16 + 2h + 1) of part Q are adjacent
        // bytes of a scale-factor atom.  Rows the TMA stores clip (>= F, or past the unit) must not be written here.
        const int pf = PACKED ? row_l / pk_g : 0, pj = PACKED ? j + (row_l & (pk_g - 1)) : 0;   // packed: frame, joint of the row
        const int64_t tok = SPATIAL  ? static_cast<int64_t>(j) + row_l
                            : PACKED ? (static_cast<int64_t>(b) * F + pf) * j_tok + pj
                                     : (static_cast<int64_t>(b) * F + r) * J + j;
        const bool live = SPATIAL ? row_l < (tail ? (F % 7) * 17 : kSpatialRows) : PACKED ? (pf < F && pj < j_tok) : r < F;
        if (live) {
          *reinterpret_cast<uint16_t*>(sf_out + op_sf_offset(tok, 2 * h, kC / 64)) = static_cast<uint16_t>(bp0 | (bp1 << 8));
          *reinterpret_cast<uint16_t*>(sf_out + op_sf_offset(tok, 16 + 2 * h, kC / 64)) = static_cast<uint16_t>(bq0 | (bq1 << 8));
        }
      } else {
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        // packed pairs: x = O inv - (v_hi + v_lo), lo = x - fp16(x) and the two e5m2 scalings as FFMA2 / FADD2 / FMUL2
        uint32_t hw[4], lw[4], a8[4], l8[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float oa = __uint_as_float(g < 4 ? o0[8 * g + 2 * e] : o1[8 * (g & 3) + 2 * e]);
          const float ob = __uint_as_float(g < 4 ? o0[8 * g + 2 * e + 1] : o1[8 * (g & 3) + 2 * e + 1]);
          float x0, x1, l0, l1;
          const ptx::f32x2 xp = ptx::fma2(ptx::pack2(oa, ob), inv2, nv[4 * g + e]);
          ptx::unpack2(xp, x0, x1);
          const __half2 h01 = __floats2half2_rn(x0, x1);
          const float2 hf = __half22float2(h01);
          const ptx::f32x2 lp = ptx::sub2(xp, ptx::pack2(hf.x, hf.y));
          hw[e] = *reinterpret_cast<const uint32_t*>(&h01);
          if (FMT == FMT_SPLIT16) {
            ptx::unpack2(lp, l0, l1);
            const __half2 l01 = __floats2half2_rn(l0, l1);
            lw[e] = *reinterpret_cast<const uint32_t*>(&l01);
          } else {
            ptx::unpack2(ptx::mul2(xp, ptx::splat2(kActHiScale)), x0, x1);
            ptx::unpack2(ptx::mul2(lp, ptx::splat2(kActLoScale)), l0, l1);
            a8[e] = op_e5m2x2(x0, x1);
            l8[e] = op_e5m2x2(l0, l1);
          }
        }
        *reinterpret_cast<uint4*>(hi_row + ((g << 4) ^ sw)) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
        if (FMT == FMT_SPLIT16) {            // lo rows: 128 B, swizzled like hi
          *reinterpret_cast<uint4*>(Stg + row_l * 128 + ((g << 4) ^ sw)) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
        } else {                             // c8: [128 rows][64 B] e5m2(x 2^-8), then [128 rows][64 B] e5m2(lo 2^4)
          *reinterpret_cast<uint2*>(Stg + row_l * 64 + g * 8) = make_uint2(a8[0] | (a8[1] << 16), a8[2] | (a8[3] << 16));
          *reinterpret_cast<uint2*>(Stg + 8192 + row_l * 64 + g * 8) = make_uint2(l8[0] | (l8[1] << 16), l8[2] | (l8[3] << 16));
        }
      }
      }
      ptx::fence_proxy_async();
      ptx::bar_sync(1 + slot, 128);          // every row is staged, and nobody still reads v_hi rows of this tile
      if (D3D_ATTN_STORE_WARP) {
        if (issuer) ptx::mbar_arrive(&bars->staged[slot]);
      } else if (issuer) {
        const CUtensorMap* mh = tail ? &tm_hi_tail : &tm_hi;
        const CUtensorMap* ms = tail ? &tm_second_tail : &tm_second;
        ptx::tma_store_4d(mh, Qs + m * kTile, h * kHd, j, m * 128, b);
        if (FMT == FMT_F4C) {                // c4 row: 256 B of P nibbles | 256 B of Q nibbles; 32 B per head and part
          ptx::tma_store_4d(ms, Stg, h * 32, j, m * 128, b);
          ptx::tma_store_4d(ms, Stg + 4096, (kC >> 1) + h * 32, j, m * 128, b);
        } else {
          ptx::tma_store_4d(ms, Stg, h * kHd, j, m * 128, b);
          if (FMT != FMT_SPLIT16) ptx::tma_store_4d(ms, Stg + 8192, kC + h * kHd, j, m * 128, b);
        }
        ptx::bulk_commit();
        ptx::bulk_wait_read_all();           // Stg / Q_m have been read: the tile has left shared memory
        ptx::mbar_arrive(&bars->stage_free[stage]);
      }
    }
    if (!D3D_ATTN_STORE_WARP && issuer) ptx::bulk_wait_all();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<kTmemCols>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Temporal mode with TWO softmax warpgroups per slot (FMT_F4C, 64 < F <= 256; round 2).
//
// ncu on the kernel above at F = 243 (profiles/r02f_full_attn_temporal.md + source page): 11 000 warp-instructions per
// 128 x 256 tile executed by FOUR warps (2750 each, strictly serial: max pass, exp2 pass, "- V", epilogue), 1.9 issued
// instructions per cycle and SM with two warps per scheduler, MUFU 35 % busy, DRAM 49 %: the tile time is the length of
// one thread's instruction stream, not a throughput limit.  Here a slot's 128 rows are owned by two warpgroups:
//   half h (0 / 1) takes the 32-column chunks [c0_h, c1_h) of S (c_split = ceil(n / 2)) and, in the epilogue, the 32
//   channels [32 h, 32 h + 32) of the row -- exactly one scale block of each part;
//   * row maximum: partial maxima meet in shared memory (one named barrier of the slot's 256 threads);
//   * P of chunk c is written at TMEM column  32 c0_h + 16 (c - c0_h): the start of the half's OWN S columns, so no half
//     overwrites S columns the other one still reads (the single-warpgroup layout, P contiguous from column 0, would);
//     the P.V chain takes its A operand from the two ranges;
//   * O = P.V accumulates into columns [192, 256) (NKp > 128; S chunks 6, 7 are dead once both halves arrived on p_full)
//     or [128, 192);
//   * row sums meet in shared memory behind the barrier that already guards the staging buffer.
// 640 threads: warps 0..15 softmax (warpgroup = slot * 2 + half, TMEM lane quadrant = warp & 3), 16 = TMA producer,
// 17 = MMA issuer / TMEM allocator, 18..19 idle.  96 registers at launch; control warpgroup 40, softmax warpgroups 104.
//
// MEASURED (profiles/r02o_*, r02p_*): correct (the whole GPU suite passes on it) and 23 % SLOWER than the one-warpgroup
// kernel at cfg3 (357 vs 290 ms of temporal attention per step), so it ships OFF (D3D_ATTN_WG2=1 selects it).  The two
// halves of a row share the TMEM lane quadrant and with it the SM sub-partition's MUFU unit: the exp2 pass of a tile costs
// 256 MUFU per row and sub-partition either way (2048 cycles), both halves reach it together behind the exchange barrier,
// and what the split saves in the max pass and the epilogue is less than the third 256-thread barrier per tile, the TMEM
// loads no longer issued a batch ahead (104 instead of 216 registers) and the spills cost.  What would help is MUFU
// capacity, not threads: part of the exp2 on the FMA pipes (DESIGN.md section 7).
constexpr int kTc2Threads = 640;
constexpr int kCtrlRegs2 = 40, kSoftmaxRegs2 = 104;
static_assert(4 * 128 * (kSoftmaxRegs2 - 96) <= 128 * (96 - kCtrlRegs2), "setmaxnreg pool overdrawn");

// P column (offset inside the slot) of chunk c
__device__ __forceinline__ int p_col2(int c, int c_split) { return c < c_split ? c * 16 : 32 * c_split + (c - c_split) * 16; }

template <int NCH>
__global__ void __launch_bounds__(kTc2Threads, 1)
attn_temporal_tc2_kernel(const __grid_constant__ CUtensorMap tm_qkv, const __grid_constant__ CUtensorMap tm_hi,
                         const __grid_constant__ CUtensorMap tm_second, uint8_t* __restrict__ sf_out, int F, int J,
                         int n_units, int n_mt, int NKp, int n_stage) {
  constexpr int NSLOT = 2;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int stage_bytes = 3 * n_mt * kTile;
  uint8_t* StgAll = smem + n_stage * stage_bytes;    // per slot 16 KB: [0, 4 KB) P tile, [4, 8 KB) Q tile, [8 KB, ..) exchange
  TcBars<NSLOT>* bars = reinterpret_cast<TcBars<NSLOT>*>(StgAll + NSLOT * kTile);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int kTmaWarp = 16, kMmaWarp = 17;
  const int n_local = blockIdx.x < n_units ? (n_units - 1 - static_cast<int>(blockIdx.x)) / static_cast<int>(gridDim.x) + 1 : 0;
  const int W = n_local * n_mt;
  const int n_chunks = (NKp + 31) >> 5;
  const int c_split = (n_chunks + 1) >> 1;
  const uint32_t o_col = NKp > 128 ? 192u : 128u;

  if (warp == kTmaWarp && ptx::elect_one()) {
    ptx::prefetch_tensormap(&tm_qkv);
    ptx::prefetch_tensormap(&tm_hi);
    ptx::prefetch_tensormap(&tm_second);
    for (int s = 0; s < n_stage; ++s) {
      ptx::mbar_init(&bars->full[s], 1);
      ptx::mbar_init(&bars->stage_free[s], n_mt);
    }
#pragma unroll
    for (int s = 0; s < NSLOT; ++s) {
      ptx::mbar_init(&bars->s_full[s], 1);
      ptx::mbar_init(&bars->p_full[s], 256);
      ptx::mbar_init(&bars->o_full[s], 1);
      ptx::mbar_init(&bars->tmem_free[s], 256);
      ptx::mbar_init(&bars->vlo_full[s], 1);
    }
    ptx::fence_barrier_init();
  }
  if (warp == kMmaWarp) ptx::tmem_alloc<kSlotCols * NSLOT>(&bars->tmem_base);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  if (warp == kTmaWarp) {
    // ------------------------------------------------------------------ TMA producer
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kCtrlRegs2));
    if (ptx::elect_one()) {
      for (int n = 0; n < n_local; ++n) {
        const int unit = blockIdx.x + n * gridDim.x;
        const int seq = unit >> 3, h = unit & 7;
        const int b = seq / J, j = seq - b * J;
        const int stage = n % n_stage, k = n / n_stage;
        uint8_t* Qs = smem + stage * stage_bytes;
        uint8_t* Ks = Qs + n_mt * kTile;
        uint8_t* Vs = Ks + n_mt * kTile;
        ptx::mbar_wait(&bars->stage_free[stage], (k & 1) ^ 1);
        ptx::mbar_arrive_expect_tx(&bars->full[stage], 3 * n_mt * kTile);
        for (int t = 0; t < n_mt; ++t) {
          ptx::tma_load_4d(Ks + t * kTile, &tm_qkv, &bars->full[stage], kC + h * kHd, j, t * 128, b);
          ptx::tma_load_4d(Qs + t * kTile, &tm_qkv, &bars->full[stage], h * kHd, j, t * 128, b);
          ptx::tma_load_4d(Vs + t * kTile, &tm_qkv, &bars->full[stage], 2 * kC + h * kHd, j, t * 128, b);
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------------------------------------------ MMA issuer
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kCtrlRegs2));
    if (ptx::elect_one()) {
      const uint32_t idesc_qk = ptx::make_idesc_f16(128, static_cast<uint32_t>(NKp), 0);
      const uint32_t idesc_pv = ptx::make_idesc_f16(128, kHd, 0) | (1u << 16);      // B (= V) is MN-major
      const uint32_t s0 = ptx::smem_u32(smem);
      const int n_ks = NKp >> 4;
      auto issue_pv = [&](int w) {           // O[128, 64] = P[128, NKp] (TMEM, two column ranges) . V[NKp, 64], 16 keys per MMA
        const int slot = w % NSLOT, i = w / NSLOT, stage = (w / n_mt) % n_stage;
        const uint32_t sV = s0 + stage * stage_bytes + 2 * n_mt * kTile;
        const uint32_t tcol = tmem_base + slot * kSlotCols;
        ptx::mbar_wait(&bars->p_full[slot], i & 1);
        ptx::tc_fence_after();
        for (int ks = 0; ks < n_ks; ++ks)
          ptx::mma_f16_ts(tcol + o_col, tcol + p_col2(ks >> 1, c_split) + (ks & 1) * 8, make_desc_mn_sw128(sV + ks * 2048),
                          idesc_pv, ks != 0 ? 1u : 0u);
        ptx::mma_commit(&bars->o_full[slot]);
      };
      for (int w = 0; w < W; ++w) {
        const int n = w / n_mt, m = w - n * n_mt;
        const int slot = w % NSLOT, i = w / NSLOT, stage = n % n_stage;
        const uint32_t sQ = s0 + stage * stage_bytes, sK = sQ + n_mt * kTile;
        if (m == 0) {
          ptx::mbar_wait(&bars->full[stage], (n / n_stage) & 1);
          ptx::tc_fence_after();
        }
        ptx::mbar_wait(&bars->tmem_free[slot], (i & 1) ^ 1);
        ptx::tc_fence_after();
#pragma unroll
        for (int k = 0; k < 4; ++k)
          ptx::mma_f16_ss(tmem_base + slot * kSlotCols, ptx::make_desc_k_sw128(sQ + m * kTile + k * 32),
                          ptx::make_desc_k_sw128(sK + k * 32), idesc_qk, k != 0 ? 1u : 0u);
        ptx::mma_commit(&bars->s_full[slot]);
        if (w >= NSLOT - 1) issue_pv(w - (NSLOT - 1));
      }
      for (int w = W - (NSLOT - 1); w < W; ++w)
        if (w >= 0) issue_pv(w);
    }
  } else if (warp > kMmaWarp) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kCtrlRegs2));
  } else {
    // ------------------------------------------------------------------ softmax + epilogue: thread = (query row, half)
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kSoftmaxRegs2));
    const int wg = warp >> 2, slot = wg >> 1, half = wg & 1;
    const int row_l = (warp & 3) * 32 + lane;
    const uint32_t taddr = tmem_base + slot * kSlotCols + (static_cast<uint32_t>((warp & 3) * 32) << 16);
    if (NCH > 0 && (n_chunks != NCH || F <= 32 * (NCH - 1))) __trap();
    const int c0 = half ? c_split : 0, c1 = half ? n_chunks : c_split;       // this half's chunks of S
    constexpr int kMaxHalf = NCH > 0 ? (NCH + 1) / 2 : 4;
    const int sw = (row_l & 7) << 4;
    const bool issuer = half == 0 && row_l == 0;
    uint8_t* Stg = StgAll + slot * kTile;
    float* xmax = reinterpret_cast<float*>(Stg + 8192);      // [2 halves][128 rows]
    float* xsum = xmax + 256;
    auto full = [&](int c) { return (c + 1) * 32 <= F; };
    for (int w = slot; w < W; w += NSLOT) {
      const int n = w / n_mt, m = w - n * n_mt;
      const int i = w / NSLOT, stage = n % n_stage;
      const int unit = blockIdx.x + n * gridDim.x;
      const int seq = unit >> 3, h = unit & 7;
      const int b = seq / J, j = seq - b * J;
      uint8_t* Qs = smem + stage * stage_bytes;
      const uint8_t* Vs = Qs + 2 * n_mt * kTile;
      const int r = m * 128 + row_l;
      ptx::mbar_wait(&bars->s_full[slot], i & 1);
      ptx::tc_fence_after();
      if (issuer) {      // Q_m is dead once S is complete: it receives the v_lo rows of the tile (exact "- V" term)
        ptx::mbar_arrive_expect_tx(&bars->vlo_full[slot], kTile);
        ptx::tma_load_4d(Qs + m * kTile, &tm_qkv, &bars->vlo_full[slot], 3 * kC + h * kHd, j, m * 128, b);
      }
      // ---- pass 1: maximum over this half's columns, then over the row
      uint32_t a0[32], a1[32];
      float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
      auto max_chunk = [&](const uint32_t (&rr)[32], int c) {
        if (full(c)) {
#pragma unroll
          for (int e = 0; e < 32; ++e) mx[e & 3] = fmaxf(mx[e & 3], __uint_as_float(rr[e]));
        } else {
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if (c * 32 + e < F) mx[e & 3] = fmaxf(mx[e & 3], __uint_as_float(rr[e]));
        }
      };
#pragma unroll
      for (int q = 0; q < kMaxHalf; q += 2) {
        const int c = c0 + q;
        if (c < c1) {
          ptx::tmem_ld_32x32(taddr + c * 32, a0);
          if (c + 1 < c1) ptx::tmem_ld_32x32(taddr + (c + 1) * 32, a1);
          ptx::tmem_ld_wait();
          max_chunk(a0, c);
          if (c + 1 < c1) max_chunk(a1, c + 1);
        }
      }
      const float m_own = fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3]));
      xmax[half * 128 + row_l] = m_own;
      ptx::tmem_ld_32x32(taddr + c0 * 32, a0);                   // pass 2 streams in behind the exchange barrier
      if (c0 + 1 < c1) ptx::tmem_ld_32x32(taddr + (c0 + 1) * 32, a1);
      ptx::bar_sync(1 + slot, 256);
      const float nmxs = -fmaxf(m_own, xmax[(half ^ 1) * 128 + row_l]) * kScaleLog2e;
      // ---- pass 2: P = exp2(S c - m c) as packed fp16 at the start of this half's own S columns, partial row sum
      ptx::f32x2 ls[2] = {ptx::splat2(0.f), ptx::splat2(0.f)};
      const ptx::f32x2 sc2 = ptx::splat2(kScaleLog2e), nm2 = ptx::splat2(nmxs);
      auto exp_chunk = [&](const uint32_t (&rr)[32], int c) {
        uint32_t pk[16];
        if (full(c)) {                         // warp-uniform: every chunk but the row's last one takes the unmasked form
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            float t0, t1;
            ptx::unpack2(ptx::fma2(ptx::pack2(__uint_as_float(rr[2 * e]), __uint_as_float(rr[2 * e + 1])), sc2, nm2), t0, t1);
            const float e0 = ex2_approx(t0), e1 = ex2_approx(t1);
            ls[e & 1] = ptx::add2(ls[e & 1], ptx::pack2(e0, e1));
            pk[e] = pack_f16x2(e0, e1);
          }
        } else {
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            float t0, t1;
            ptx::unpack2(ptx::fma2(ptx::pack2(__uint_as_float(rr[2 * e]), __uint_as_float(rr[2 * e + 1])), sc2, nm2), t0, t1);
            const int col = c * 32 + 2 * e;
            const float e0 = col < F ? ex2_approx(t0) : 0.f;
            const float e1 = col + 1 < F ? ex2_approx(t1) : 0.f;
            ls[e & 1] = ptx::add2(ls[e & 1], ptx::pack2(e0, e1));
            pk[e] = pack_f16x2(e0, e1);
          }
        }
        ptx::tmem_st_32x16(taddr + 32 * c0 + (c - c0) * 16, pk);
      };
#pragma unroll
      for (int q = 0; q < kMaxHalf; q += 2) {
        const int c = c0 + q;
        if (c < c1) {
          if (q > 0) {
            ptx::tmem_ld_32x32(taddr + c * 32, a0);
            if (c + 1 < c1) ptx::tmem_ld_32x32(taddr + (c + 1) * 32, a1);
          }
          ptx::tmem_ld_wait();
          exp_chunk(a0, c);
          if (c + 1 < c1) exp_chunk(a1, c + 1);
        }
      }
      ptx::tmem_st_wait();
      xsum[half * 128 + row_l] = row_sum(ls);
      ptx::tc_fence_before();
      ptx::mbar_arrive(&bars->p_full[slot]);

      // ---- while the P.V chain runs: this half's 32 channels of the exact "- V" term
      ptx::mbar_wait(&bars->vlo_full[slot], i & 1);
      const uint32_t hi_row = ptx::smem_u32(Qs + m * kTile + row_l * 128);   // v_lo row in, hi row out
      const uint32_t v_row = ptx::smem_u32(Vs) + static_cast<uint32_t>(r) * 128;
      ptx::f32x2 nv[16];
      {
        uint4 vh[4], vl[4];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          vh[g] = ptx::lds128(v_row + (((half * 4 + g) << 4) ^ sw));
          vl[g] = ptx::lds128(hi_row + (((half * 4 + g) << 4) ^ sw));
        }
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const uint32_t vhw[4] = {vh[g].x, vh[g].y, vh[g].z, vh[g].w};
          const uint32_t vlw[4] = {vl[g].x, vl[g].y, vl[g].z, vl[g].w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&vhw[e]));
            const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&vlw[e]));
            float s0, s1;
            ptx::unpack2(ptx::add2(ptx::pack2(a.x, a.y), ptx::pack2(c.x, c.y)), s0, s1);
            nv[4 * g + e] = ptx::pack2(-s0, -s1);
          }
        }
      }
      // ---- this half's 32 columns of O out of TMEM, then the slot is free for the next S
      ptx::mbar_wait(&bars->o_full[slot], i & 1);
      ptx::tc_fence_after();
      uint32_t o0[32];
      ptx::tmem_ld_32x32(taddr + o_col + half * 32, o0);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(&bars->tmem_free[slot]);

      // ---- epilogue: out = O / l - (v_hi + v_lo): one scale block of each part per half
      ptx::bar_sync(1 + slot, 256);          // the previous tile's stores have read Stg; both partial row sums are visible
      const ptx::f32x2 inv2 = ptx::splat2(rcp_approx(xsum[row_l] + xsum[128 + row_l]));
      float ax = 0.f, al = 0.f;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint32_t hw[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          float x0, x1;
          ptx::unpack2(ptx::fma2(ptx::pack2(__uint_as_float(o0[8 * g + 2 * e]), __uint_as_float(o0[8 * g + 2 * e + 1])), inv2,
                                 nv[4 * g + e]), x0, x1);
          const __half2 h01 = __floats2half2_rn(x0, x1);
          const float2 hf = __half22float2(h01);
          hw[e] = *reinterpret_cast<const uint32_t*>(&h01);
          ax = fmaxf(ax, fmaxf(fabsf(x0), fabsf(x1)));
          al = fmaxf(al, fmaxf(fabsf(x0 - hf.x), fabsf(x1 - hf.y)));
          o0[8 * g + 2 * e] = __float_as_uint(x0);
          o0[8 * g + 2 * e + 1] = __float_as_uint(x1);
        }
        ptx::sts128(hi_row + (((half * 4 + g) << 4) ^ sw), make_uint4(hw[0], hw[1], hw[2], hw[3]));
      }
      const uint32_t bp = op_ue8m0_of(ax), bq = op_ue8m0_of(al);
      const ptx::f32x2 ip = ptx::splat2(op_ue8m0_inv(bp)), iq = ptx::splat2(op_ue8m0_inv(bq));
      uint32_t pw[4], qw[4];
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint32_t pa = 0, qa = 0;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float x0 = __uint_as_float(o0[8 * g + 2 * e]), x1 = __uint_as_float(o0[8 * g + 2 * e + 1]);
          const float2 hf = __half22float2(__floats2half2_rn(x0, x1));
          float q0, q1, l0, l1;
          ptx::unpack2(ptx::mul2(ptx::pack2(x0, x1), ip), q0, q1);
          ptx::unpack2(ptx::mul2(ptx::sub2(ptx::pack2(x0, x1), ptx::pack2(hf.x, hf.y)), iq), l0, l1);
          pa |= op_e2m1x2(q0, q1) << (8 * e);
          qa |= op_e2m1x2(l0, l1) << (8 * e);
        }
        pw[g] = pa; qw[g] = qa;
      }
      {
        const uint32_t st = ptx::smem_u32(Stg) + row_l * 32 + half * 16;     // [128 rows][32 B] P tile, then the Q tile
        ptx::sts128(st, make_uint4(pw[0], pw[1], pw[2], pw[3]));
        ptx::sts128(st + 4096, make_uint4(qw[0], qw[1], qw[2], qw[3]));
      }
      if (r < F) {       // rows the TMA stores clip must not leave scale bytes either
        const int64_t tok = (static_cast<int64_t>(b) * F + r) * J + j;
        sf_out[op_sf_offset(tok, 2 * h + half, kC / 64)] = static_cast<uint8_t>(bp);
        sf_out[op_sf_offset(tok, 16 + 2 * h + half, kC / 64)] = static_cast<uint8_t>(bq);
      }
      ptx::fence_proxy_async();
      ptx::bar_sync(1 + slot, 256);          // every row is staged, and nobody still reads v_hi rows of this tile
      if (issuer) {
        ptx::tma_store_4d(&tm_hi, Qs + m * kTile, h * kHd, j, m * 128, b);
        ptx::tma_store_4d(&tm_second, Stg, h * 32, j, m * 128, b);
        ptx::tma_store_4d(&tm_second, Stg + 4096, (kC >> 1) + h * 32, j, m * 128, b);
        ptx::bulk_commit();
        ptx::bulk_wait_read_all();
        ptx::mbar_arrive(&bars->stage_free[stage]);
      }
    }
    if (issuer) ptx::bulk_wait_all();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<kSlotCols * NSLOT>(tmem_base);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn query_encode_tiled() {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  return (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) ? reinterpret_cast<EncodeTiledFn>(fn) : nullptr;
}

int encode_rank4(CUtensorMap* out, void* base, CUtensorMapDataType dt, const cuuint64_t (&dims)[4],
                 const cuuint64_t (&strides)[3], const cuuint32_t (&box)[4], CUtensorMapSwizzle swz) {
  // fetched once; a function-local static is initialised thread-safely when handles are created concurrently
  static const EncodeTiledFn encode = query_encode_tiled();
  if (!encode) return -1;
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = encode(out, dt, 4, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : -static_cast<int>(r) - 1000;
}

// [B, F, J, row] token-major array viewed as a 4-D tensor (channel, j, f, b); box = {64 channels, 1, 128 frames, 1}
// box_j > 1 (packed mode, F <= 64): box = {box0 channels, box_j joints, 128 / box_j frames, 1}, rows land as f * box_j + jj
int encode_tokens_4d(CUtensorMap* out, void* base, CUtensorMapDataType dt, int elem_bytes, int64_t row_elems, int J,
                     int F, int64_t B, CUtensorMapSwizzle swz, int box0 = 64, int box_j = 1) {
  const cuuint64_t row_bytes = static_cast<cuuint64_t>(row_elems) * elem_bytes;
  const cuuint64_t dims[4] = {static_cast<cuuint64_t>(row_elems), static_cast<cuuint64_t>(J), static_cast<cuuint64_t>(F),
                              static_cast<cuuint64_t>(B)};
  const cuuint64_t strides[3] = {row_bytes, row_bytes * J, row_bytes * J * F};
  const cuuint32_t box[4] = {static_cast<cuuint32_t>(box0), static_cast<cuuint32_t>(box_j),
                             static_cast<cuuint32_t>(128 / box_j), 1};
  return encode_rank4(out, base, dt, dims, strides, box, swz);
}

// The same array as a plain [tokens, row] matrix (rank 4 with two unit dimensions, so that the kernel's 4-D TMA
// instructions serve both modes); box = {64 channels, box_rows tokens, 1, 1}
int encode_tokens_2d(CUtensorMap* out, void* base, CUtensorMapDataType dt, int elem_bytes, int64_t row_elems,
                     int64_t tokens, int box_rows, CUtensorMapSwizzle swz, int box0 = 64) {
  const cuuint64_t row_bytes = static_cast<cuuint64_t>(row_elems) * elem_bytes;
  const cuuint64_t dims[4] = {static_cast<cuuint64_t>(row_elems), static_cast<cuuint64_t>(tokens), 1, 1};
  const cuuint64_t strides[3] = {row_bytes, row_bytes * tokens, row_bytes * tokens};
  const cuuint32_t box[4] = {static_cast<cuuint32_t>(box0), static_cast<cuuint32_t>(box_rows), 1, 1};
  return encode_rank4(out, base, dt, dims, strides, box, swz);
}

inline int tc_stages(int n_mt) { return n_mt == 1 ? 4 : 2; }
template <int NSLOT>
int tc_smem_bytes(int n_mt) {
  return tc_stages(n_mt) * 3 * n_mt * kTile + NSLOT * (NSLOT == 2 ? kTile : 8192) + static_cast<int>(sizeof(TcBars<NSLOT>)) +
         1024 /*alignment slack*/;
}

}  // namespace

// D3D_ATTN_SLOTS = 3: three 128-column TMEM slots / softmax warpgroups in the single-tile modes (spatial, packed temporal)
inline bool three_slots() {
  const char* v = getenv("D3D_ATTN_SLOTS");
  return v && *v == '3';
}
inline int packed_group(int F) { return F <= 32 ? 4 : (F <= 64 ? 2 : 1); }     // joints per 128-row tile

int make_attn_tc_maps(AttnTcMaps* maps, const __half* qkv, __half* o_hi, __half* o_second, int fmt, int F, int J,
                      int64_t max_clips) {
  const int G = packed_group(F);
  if (encode_tokens_4d(&maps->qkv, const_cast<__half*>(qkv), CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, kQkvRow, J, F, max_clips,
                       CU_TENSOR_MAP_SWIZZLE_128B, 64, G))
    return -1;
  if (encode_tokens_4d(&maps->o_hi, o_hi, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, kC, J, F, max_clips,
                       CU_TENSOR_MAP_SWIZZLE_128B, 64, G))
    return -1;
  if (fmt == FMT_F8C)
    return encode_tokens_4d(&maps->o_second, o_second, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, 2 * kC, J, F, max_clips,
                            CU_TENSOR_MAP_SWIZZLE_NONE, 64, G);
  if (fmt == FMT_F4C)       // c4 rows of K = 512 bytes; {32 B x 128 rows} boxes (one head of one part)
    return encode_tokens_4d(&maps->o_second, o_second, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, kC, J, F, max_clips,
                            CU_TENSOR_MAP_SWIZZLE_NONE, 32, G);
  return encode_tokens_4d(&maps->o_second, o_second, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, kC, J, F, max_clips,
                          CU_TENSOR_MAP_SWIZZLE_128B, 64, G);
}

int make_attn_tc_maps_spatial(AttnTcMaps* maps, const __half* qkv, __half* o_hi, __half* o_second, int fmt,
                              int64_t tokens, int F) {
  const int tail_rows = (F % 7) ? (F % 7) * 17 : kSpatialRows;
  if (encode_tokens_2d(&maps->o_hi_tail, o_hi, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, kC, tokens, tail_rows,
                       CU_TENSOR_MAP_SWIZZLE_128B))
    return -1;
  if (fmt == FMT_F8C   ? encode_tokens_2d(&maps->o_second_tail, o_second, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, 2 * kC, tokens,
                                          tail_rows, CU_TENSOR_MAP_SWIZZLE_NONE)
      : fmt == FMT_F4C ? encode_tokens_2d(&maps->o_second_tail, o_second, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, kC, tokens,
                                          tail_rows, CU_TENSOR_MAP_SWIZZLE_NONE, 32)
                       : encode_tokens_2d(&maps->o_second_tail, o_second, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, kC, tokens,
                                          tail_rows, CU_TENSOR_MAP_SWIZZLE_128B))
    return -1;
  // loads: 128-row boxes (rows beyond the 119 of a unit are read but masked); stores: 119-row boxes
  if (encode_tokens_2d(&maps->qkv, const_cast<__half*>(qkv), CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, kQkvRow, tokens, 128,
                       CU_TENSOR_MAP_SWIZZLE_128B))
    return -1;
  if (encode_tokens_2d(&maps->o_hi, o_hi, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, kC, tokens, kSpatialRows,
                       CU_TENSOR_MAP_SWIZZLE_128B))
    return -1;
  if (fmt == FMT_F8C)
    return encode_tokens_2d(&maps->o_second, o_second, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, 2 * kC, tokens, kSpatialRows,
                            CU_TENSOR_MAP_SWIZZLE_NONE);
  if (fmt == FMT_F4C)
    return encode_tokens_2d(&maps->o_second, o_second, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, kC, tokens, kSpatialRows,
                            CU_TENSOR_MAP_SWIZZLE_NONE, 32);
  return encode_tokens_2d(&maps->o_second, o_second, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, kC, tokens, kSpatialRows,
                          CU_TENSOR_MAP_SWIZZLE_128B);
}

cudaError_t configure_attention_tc() {
  cudaError_t e;
#define D3D_CFG_TC(FMT_, NCH_, SP_)                                                                                       \
  if ((e = cudaFuncSetAttribute(attn_temporal_tc_kernel<FMT_, 2, NCH_, SP_>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                tc_smem_bytes<2>(2))) != cudaSuccess)                                                    \
    return e;
  D3D_CFG_TC(FMT_SPLIT16, 0, false) D3D_CFG_TC(FMT_F8C, 0, false) D3D_CFG_TC(FMT_SPLIT16, 3, false)
  D3D_CFG_TC(FMT_F8C, 3, false) D3D_CFG_TC(FMT_SPLIT16, 8, false) D3D_CFG_TC(FMT_F8C, 8, false)
  D3D_CFG_TC(FMT_SPLIT16, 0, true) D3D_CFG_TC(FMT_F8C, 0, true)
  D3D_CFG_TC(FMT_F4C, 0, false) D3D_CFG_TC(FMT_F4C, 3, false) D3D_CFG_TC(FMT_F4C, 8, false) D3D_CFG_TC(FMT_F4C, 0, true)
#undef D3D_CFG_TC
  if ((e = cudaFuncSetAttribute(attn_temporal_tc_kernel<FMT_F4C, 3, 0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                tc_smem_bytes<3>(1))) != cudaSuccess)
    return e;
  if ((e = cudaFuncSetAttribute(attn_temporal_tc_kernel<FMT_F4C, 3, 0, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                tc_smem_bytes<3>(1))) != cudaSuccess)
    return e;
  for (auto kern : {attn_temporal_tc2_kernel<8>, attn_temporal_tc2_kernel<3>, attn_temporal_tc2_kernel<0>})
    if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem_bytes<2>(2))) != cudaSuccess) return e;
#define D3D_CFG_PK(FMT_)                                                                                                     \
  if ((e = cudaFuncSetAttribute(attn_temporal_tc_kernel<FMT_, 2, 0, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                tc_smem_bytes<2>(1))) != cudaSuccess)                                                        \
    return e;
  D3D_CFG_PK(FMT_SPLIT16) D3D_CFG_PK(FMT_F8C) D3D_CFG_PK(FMT_F4C)
#undef D3D_CFG_PK
  return cudaSuccess;
}

cudaError_t launch_attn_temporal_tc(const AttnTcMaps& maps, const __half* qkv, uint8_t* o_sf, int fmt, int B, int F, int J,
                                    int num_sms, cudaStream_t st, int wg2) {
  if (B <= 0) return cudaSuccess;
  if (F < 1 || F > 256) return cudaErrorInvalidValue;
  if (fmt == FMT_F4C && !o_sf) return cudaErrorInvalidValue;
  if (F <= 64) {
    // packed mode: G joints of one (clip, head) per 128-row tile; the maps were built with {.., G, 128 / G, 1} boxes
    const int G = packed_group(F), JG = (J + G - 1) / G;
    const int64_t units64 = static_cast<int64_t>(B) * JG * kHeads;
    if (units64 > 0x7fffffff) return cudaErrorInvalidValue;
    const int n_units = static_cast<int>(units64);
    const int grid = n_units < num_sms ? n_units : num_sms;
    const int smem = tc_smem_bytes<2>(1);
#define D3D_LAUNCH_PK(FMT_)                                                                   \
  attn_temporal_tc_kernel<FMT_, 2, 0, false, true><<<grid, kTcThreads, smem, st>>>(           \
      maps.qkv, maps.o_hi, maps.o_second, maps.o_hi, maps.o_second, o_sf, F, JG, n_units, 1, 128, tc_stages(1), G, J)
    if (fmt == FMT_F4C && three_slots())
      attn_temporal_tc_kernel<FMT_F4C, 3, 0, false, true><<<grid, 512, tc_smem_bytes<3>(1), st>>>(
          maps.qkv, maps.o_hi, maps.o_second, maps.o_hi, maps.o_second, o_sf, F, JG, n_units, 1, 128, tc_stages(1), G, J);
    else if (fmt == FMT_F4C) D3D_LAUNCH_PK(FMT_F4C);
    else if (fmt == FMT_F8C) D3D_LAUNCH_PK(FMT_F8C);
    else D3D_LAUNCH_PK(FMT_SPLIT16);
#undef D3D_LAUNCH_PK
    return cudaGetLastError();
  }
  const int n_mt = (F + 127) / 128;
  const int NKp = (F + 15) / 16 * 16;
  const int n_units = B * J * kHeads;
  const int n_chunks = (NKp + 31) / 32;
  const int nch = (n_chunks == 8 && F > 224) ? 8 : ((n_chunks == 3 && F > 64) ? 3 : 0);   // F = 243 / 81 specialisations
  const int grid = n_units < num_sms ? n_units : num_sms;
  const int smem = tc_smem_bytes<2>(n_mt);
#define D3D_LAUNCH_TC(FMT_, NCH_)                                                                               \
  attn_temporal_tc_kernel<FMT_, 2, NCH_, false><<<grid, kTcThreads, smem, st>>>(                      \
      maps.qkv, maps.o_hi, maps.o_second, maps.o_hi, maps.o_second, o_sf, F, J, n_units, n_mt, NKp, tc_stages(n_mt))
  if (fmt == FMT_F4C && wg2) {
    // two softmax warpgroups per slot (D3D_ATTN_WG2=0: the one-warpgroup kernel)
    if (!o_sf) return cudaErrorInvalidValue;
#define D3D_LAUNCH_TC2(NCH_)                                                       \
  attn_temporal_tc2_kernel<NCH_><<<grid, kTc2Threads, smem, st>>>(maps.qkv, maps.o_hi, maps.o_second, o_sf, F, J, n_units, \
                                                                   n_mt, NKp, tc_stages(n_mt))
    if (nch == 8) D3D_LAUNCH_TC2(8); else if (nch == 3) D3D_LAUNCH_TC2(3); else D3D_LAUNCH_TC2(0);
#undef D3D_LAUNCH_TC2
  } else if (fmt == FMT_F4C) {
    if (!o_sf) return cudaErrorInvalidValue;
    if (nch == 8) D3D_LAUNCH_TC(FMT_F4C, 8); else if (nch == 3) D3D_LAUNCH_TC(FMT_F4C, 3); else D3D_LAUNCH_TC(FMT_F4C, 0);
  } else if (fmt == FMT_F8C) {
    if (nch == 8) D3D_LAUNCH_TC(FMT_F8C, 8); else if (nch == 3) D3D_LAUNCH_TC(FMT_F8C, 3); else D3D_LAUNCH_TC(FMT_F8C, 0);
  } else {
    if (nch == 8) D3D_LAUNCH_TC(FMT_SPLIT16, 8); else if (nch == 3) D3D_LAUNCH_TC(FMT_SPLIT16, 3); else D3D_LAUNCH_TC(FMT_SPLIT16, 0);
  }
#undef D3D_LAUNCH_TC
  return cudaGetLastError();
}

// Spatial mode (J == 17): units of (clip, 7-frame group, head)
cudaError_t launch_attn_spatial_tc(const AttnTcMaps& maps, uint8_t* o_sf, int fmt, int B, int F, int num_sms,
                                   cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  const int G = (F + 6) / 7;
  const int64_t units64 = static_cast<int64_t>(B) * G * kHeads;
  if (units64 > 0x7fffffff) return cudaErrorInvalidValue;
  const int n_units = static_cast<int>(units64);
  const int grid = n_units < num_sms ? n_units : num_sms;
  const int smem = tc_smem_bytes<2>(1);
  if (fmt == FMT_F4C && three_slots()) {
    if (!o_sf) return cudaErrorInvalidValue;
    attn_temporal_tc_kernel<FMT_F4C, 3, 0, true><<<grid, 512, tc_smem_bytes<3>(1), st>>>(
        maps.qkv, maps.o_hi, maps.o_second, maps.o_hi_tail, maps.o_second_tail, o_sf, F, G, n_units, 1, 128, tc_stages(1));
  } else if (fmt == FMT_F4C) {
    if (!o_sf) return cudaErrorInvalidValue;
    attn_temporal_tc_kernel<FMT_F4C, 2, 0, true><<<grid, kTcThreads, smem, st>>>(
        maps.qkv, maps.o_hi, maps.o_second, maps.o_hi_tail, maps.o_second_tail, o_sf, F, G, n_units, 1, 128, tc_stages(1));
  } else if (fmt == FMT_F8C) {
    attn_temporal_tc_kernel<FMT_F8C, 2, 0, true><<<grid, kTcThreads, smem, st>>>(
        maps.qkv, maps.o_hi, maps.o_second, maps.o_hi_tail, maps.o_second_tail, o_sf, F, G, n_units, 1, 128, tc_stages(1));
  } else {
    attn_temporal_tc_kernel<FMT_SPLIT16, 2, 0, true><<<grid, kTcThreads, smem, st>>>(
        maps.qkv, maps.o_hi, maps.o_second, maps.o_hi_tail, maps.o_second_tail, o_sf, F, G, n_units, 1, 128, tc_stages(1));
  }
  return cudaGetLastError();
}

}  // namespace d3d
