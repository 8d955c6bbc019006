// GRAND attention cores (MODEL:76-83) on tensor cores, reading the packed fp16 tensor written by the qkv GEMM
// epilogue (EPI_QKV16):  row of token t = q(512) | k(512) | v_hi(512) | v_lo(512) halves, channel inside each
// 512 = head*64 + d, token = (b*F + f)*J + j.
//
//     O = softmax(Q K^T * hd^-0.5) V  -  V[query]            ((P - I) V == P V - V, SURVEY.md K12)
//
// Q.K^T and P.V are single fp16 passes with fp32 accumulation (mma.sync.m16n8k16); the subtracted V row is
// taken as v_hi + v_lo, i.e. exact to ~2^-22, because rounding it to fp16 was the dominant error term of an
// all-fp16 attention in the CPU precision emulation (tools/precision_probe.py): with the exact "- V" the
// F=243 sampler stays at max-abs 1.5e-3 (bar 1e-2) and |dMPJPE| 2.5e-6 (bar 1e-4).
//
//   attn_temporal_h16_kernel  G-tattn: one CTA per (clip b, joint j, head); the F frames of that joint are
//       gathered with a stride of J tokens (the reference's transpose copies, MODEL:121,133, never happen).
//       K and V of the sequence are parked in shared memory with cp.async; each warp owns 16-query tiles and
//       sweeps the keys in 64-key chunks with an online softmax (exp2 domain).
//   attn_spatial_h16_kernel   G-sattn: one CTA per frame, one warp per head; the 17 joints are padded to
//       2 x 16 query rows / 24 keys, P stays in registers, the output is staged in shared memory so that every
//       global store is a full 128-byte row segment.
//
// Output: token-major [T, 512] (heads merged, MODEL:83) as the split-fp16 A operand of the proj GEMM, or fp32.
#include "kernels.cuh"
#include "operand.cuh"

namespace d3d {
namespace {

// mma.sync kernels (validation / bring-up modes): built for C = 512 only
constexpr int kC = Width<512>::kC, kHd = Width<512>::kHd, kQkvRow = Width<512>::kQkvRow;

constexpr int KS = 72;            // smem row stride in halves (144 B: ldmatrix rows hit distinct banks)
constexpr float kScaleLog2e = 0.125f * 1.4426950408889634f;   // head_dim ** -0.5 (MODEL:65) in the exp2 domain

__device__ __forceinline__ uint32_t pack2(__half a, __half b) {
  return static_cast<uint32_t>(__half_as_ushort(a)) | (static_cast<uint32_t>(__half_as_ushort(b)) << 16);
}
__device__ __forceinline__ uint32_t pack2f(float x, float y) { return pack2(__float2half_rn(x), __float2half_rn(y)); }
__device__ __forceinline__ void split2(float x, float y, uint32_t& hi, uint32_t& lo) {
  const __half hx = __float2half_rn(x), hy = __float2half_rn(y);
  hi = pack2(hx, hy);
  lo = pack2(__float2half_rn(x - __half2float(hx)), __float2half_rn(y - __half2float(hy)));
}
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cp_async16(uint32_t smem_addr, const void* gptr) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(gptr) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
// wait until at most n (0..3) of the most recently committed groups are still in flight
__device__ __forceinline__ void cp_async_wait_pending(int n) {
  switch (n) {
    case 0: asm volatile("cp.async.wait_group 0;" ::: "memory"); break;
    case 1: asm volatile("cp.async.wait_group 1;" ::: "memory"); break;
    case 2: asm volatile("cp.async.wait_group 2;" ::: "memory"); break;
    default: asm volatile("cp.async.wait_group 3;" ::: "memory"); break;
  }
}
// MUFU approximations (rel. error ~2^-22): the library exp2f / IEEE division carry slow-path branches
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ------------------------------------------------------------------------------------------ temporal
constexpr int kTStgRow = 272;                     // bytes per staged output row (256 + 16: conflict-free 4-byte writes)
constexpr int kTStgWarp = 16 * kTStgRow;          // one 16-query tile per warp

template <int FMT>
__global__ void __launch_bounds__(256, 2)
attn_temporal_h16_kernel(const __half* __restrict__ qkv, __half* __restrict__ o_hi, __half* __restrict__ o_lo,
                         float* __restrict__ o_f32, int F, int J, int NK) {
  extern __shared__ __align__(16) __half smh[];
  __half* Ks = smh;
  __half* Vs = Ks + NK * KS;
  uint8_t* stg = reinterpret_cast<uint8_t*>(Vs + NK * KS) + (threadIdx.x >> 5) * kTStgWarp;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const int head = blockIdx.y;
  const int64_t seq = blockIdx.x;                                   // b * J + j
  const int64_t tok0 = (seq / J) * (static_cast<int64_t>(F) * J) + (seq % J);
  const __half* base = qkv + head * kHd;                            // + tok * kQkvRow (+ 512 k, + 1024 v_hi, + 1536 v_lo)

  // ---- stage K, V_hi rows of the sequence (128 B each) with cp.async, one commit group per 64-key chunk so that
  //      the first q-tile sweep can start on chunk 0 while chunks 1..3 are still in flight; zero the rows beyond F
  const uint32_t sK = static_cast<uint32_t>(__cvta_generic_to_shared(Ks));
  const uint32_t sV = static_cast<uint32_t>(__cvta_generic_to_shared(Vs));
  const int n_chunks = NK >> 6;
  for (int kc = 0; kc < n_chunks; ++kc) {
    for (int i = threadIdx.x; i < 64 * 16; i += blockDim.x) {
      const int r = (kc << 6) + (i >> 4), c = i & 15;
      const bool is_v = c >= 8;
      const int c8 = c & 7;
      const uint32_t dst = (is_v ? sV : sK) + static_cast<uint32_t>((r * KS + c8 * 8) * 2);
      if (r < F) {
        const __half* src = base + static_cast<size_t>(tok0 + static_cast<int64_t>(r) * J) * kQkvRow +
                            (is_v ? 2 * kC : kC) + c8 * 8;
        cp_async16(dst, src);
      } else {
        asm volatile("st.shared.v4.u32 [%0], {%1,%1,%1,%1};" ::"r"(dst), "r"(0u) : "memory");
      }
    }
    cp_async_commit();
  }

  const int g = lane >> 2, q4 = lane & 3;
  // ldmatrix lane -> row/col offsets
  const int k_key = (lane & 7) + ((lane >> 4) << 3);     // K (B operand, non-trans): key offset within 16
  const int k_d = ((lane >> 3) & 1) << 3;                //                            d offset (0 / 8)
  const int v_key = (lane & 7) + (((lane >> 3) & 1) << 3);   // V (trans): key offset within 16
  const int v_d = (lane >> 4) << 3;                          //            d offset (0 / 8)

  const int n_qt = (F + 15) >> 4;
  bool first_sweep = true;        // every warp owns >= 1 q-tile (launch: warps = min(n_qt, 8)), so the syncs below are uniform
  for (int qt = warp; qt < n_qt; qt += nwarps) {
    const int q0 = qt << 4;
    const int r0 = q0 + g, r1 = r0 + 8;
    {
      // The finalize step reads this tile's v_lo rows and the next sweep this warp's next Q tile straight from global
      // (ncu: their exposed latency was ~17 % of the stall samples): pull those 128-byte rows into L2 now.
      const int pr = (lane < 16 ? q0 : q0 + 16 * nwarps) + (lane & 15);
      if (pr < F)
        prefetch_l2(base + static_cast<size_t>(tok0 + static_cast<int64_t>(pr) * J) * kQkvRow + (lane < 16 ? 3 * kC : 0));
    }
    // ---- Q fragments (A operand) straight from global: fp16 pairs
    uint32_t qa[4][4];
    {
      const __half* p0 = base + static_cast<size_t>(tok0 + static_cast<int64_t>(r0 < F ? r0 : 0) * J) * kQkvRow;
      const __half* p1 = base + static_cast<size_t>(tok0 + static_cast<int64_t>(r1 < F ? r1 : 0) * J) * kQkvRow;
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        const int c = ks * 16 + 2 * q4;
        qa[ks][0] = r0 < F ? *reinterpret_cast<const uint32_t*>(p0 + c) : 0u;
        qa[ks][1] = r1 < F ? *reinterpret_cast<const uint32_t*>(p1 + c) : 0u;
        qa[ks][2] = r0 < F ? *reinterpret_cast<const uint32_t*>(p0 + c + 8) : 0u;
        qa[ks][3] = r1 < F ? *reinterpret_cast<const uint32_t*>(p1 + c + 8) : 0u;
      }
    }
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
    float o[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) { o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f; }

    for (int kc = 0; kc < n_chunks; ++kc) {
      if (first_sweep) {            // chunk kc of K / V has landed for every thread of the CTA
        cp_async_wait_pending(n_chunks - 1 - kc);
        __syncthreads();
      }
      const int key0 = kc << 6;
      float s[8][4];
#pragma unroll
      for (int i = 0; i < 8; ++i) { s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f; }
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
        for (int np = 0; np < 4; ++np) {
          const uint32_t off = static_cast<uint32_t>(((key0 + np * 16 + k_key) * KS + ks * 16 + k_d) * 2);
          uint32_t b[4];
          ldsm_x4(sK + off, b);
          mma16816(s[2 * np], qa[ks], b[0], b[1]);
          mma16816(s[2 * np + 1], qa[ks], b[2], b[3]);
        }
      }
      // ---- scale (exp2 domain), mask, online softmax
      float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int key = key0 + nt * 8 + 2 * q4 + (e & 1);
          const float v = key < F ? s[nt][e] * kScaleLog2e : -INFINITY;
          s[nt][e] = v;
          if (e < 2) mx0 = fmaxf(mx0, v); else mx1 = fmaxf(mx1, v);
        }
      }
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);      // finite: every chunk holds >= 1 valid key
      const float c0 = ex2_approx(m0 - mn0), c1 = ex2_approx(m1 - mn1);      // exp2(-inf) = 0 on the first chunk
      m0 = mn0; m1 = mn1;
      float rs0 = 0.f, rs1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        s[nt][0] = ex2_approx(s[nt][0] - mn0); s[nt][1] = ex2_approx(s[nt][1] - mn0);
        s[nt][2] = ex2_approx(s[nt][2] - mn1); s[nt][3] = ex2_approx(s[nt][3] - mn1);
        rs0 += s[nt][0] + s[nt][1];
        rs1 += s[nt][2] + s[nt][3];
      }
      l0 = l0 * c0 + rs0;
      l1 = l1 * c1 + rs1;
#pragma unroll
      for (int i = 0; i < 8; ++i) { o[i][0] *= c0; o[i][1] *= c0; o[i][2] *= c1; o[i][3] *= c1; }
      // ---- O += P V
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        uint32_t pa[4];
        pa[0] = pack2f(s[2 * kk][0], s[2 * kk][1]);
        pa[1] = pack2f(s[2 * kk][2], s[2 * kk][3]);
        pa[2] = pack2f(s[2 * kk + 1][0], s[2 * kk + 1][1]);
        pa[3] = pack2f(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
        for (int dp = 0; dp < 4; ++dp) {
          const uint32_t off = static_cast<uint32_t>(((key0 + kk * 16 + v_key) * KS + dp * 16 + v_d) * 2);
          uint32_t vb[4];
          ldsm_x4_t(sV + off, vb);
          mma16816(o[2 * dp], pa, vb[0], vb[1]);
          mma16816(o[2 * dp + 1], pa, vb[2], vb[3]);
        }
      }
    }
    first_sweep = false;
    // ---- finalize: out = O / l - V[query],  V[query] = v_hi (smem) + v_lo (global).  The 16 x 64 tile is staged
    //      per warp (row = 128 B hi | 128 B second part, or 256 B fp32) and written with 16-byte stores.
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float i0 = rcp_approx(l0), i1 = rcp_approx(l1);
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int r = half ? r1 : r0;
      if (r >= F) continue;
      const float inv = half ? i1 : i0;
      const int64_t tok = tok0 + static_cast<int64_t>(r) * J;
      const __half* vlo = base + static_cast<size_t>(tok) * kQkvRow + 3 * kC;
      uint8_t* srow = stg + (g + 8 * half) * kTStgRow;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const int d = nt * 8 + 2 * q4;
        const __half2 vh = *reinterpret_cast<const __half2*>(Vs + r * KS + d);
        const __half2 vl = *reinterpret_cast<const __half2*>(vlo + d);
        const float x0 = o[nt][2 * half] * inv - (__low2float(vh) + __low2float(vl));
        const float x1 = o[nt][2 * half + 1] * inv - (__high2float(vh) + __high2float(vl));
        if (o_f32) {
          *reinterpret_cast<float2*>(srow + d * 4) = make_float2(x0, x1);
        } else if (FMT == FMT_SPLIT16) {
          uint32_t hh, ll;
          split2(x0, x1, hh, ll);
          *reinterpret_cast<uint32_t*>(srow + d * 2) = hh;
          *reinterpret_cast<uint32_t*>(srow + 128 + d * 2) = ll;
        } else {      // hi | e5m2(x 2^-8) (64 B) | e5m2(lo 2^4) (64 B)
          const __half h0 = __float2half_rn(x0), h1 = __float2half_rn(x1);
          *reinterpret_cast<uint32_t*>(srow + d * 2) = pack2(h0, h1);
          *reinterpret_cast<uint16_t*>(srow + 128 + d) =
              static_cast<uint16_t>(op_e5m2x2(x0 * kActHiScale, x1 * kActHiScale));
          *reinterpret_cast<uint16_t*>(srow + 192 + d) = static_cast<uint16_t>(
              op_e5m2x2((x0 - __half2float(h0)) * kActLoScale, (x1 - __half2float(h1)) * kActLoScale));
        }
      }
    }
    __syncwarp();
    uint4 vals[8];
#pragma unroll
    for (int it = 0; it < 8; ++it) {                      // all shared loads first (distinct registers), then the stores
      const int idx = it * 32 + lane;
      vals[it] = *reinterpret_cast<const uint4*>(stg + (idx >> 4) * kTStgRow + (idx & 15) * 16);
    }
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int idx = it * 32 + lane;
      const int rr = idx >> 4, c = idx & 15;              // staged row, 16-byte chunk
      const int r = q0 + rr;
      if (r < F) {
        const uint4 val = vals[it];
        const size_t tok = static_cast<size_t>(tok0 + static_cast<int64_t>(r) * J);
        if (o_f32) {
          *reinterpret_cast<uint4*>(o_f32 + tok * kC + head * kHd + c * 4) = val;
        } else if (c < 8) {
          *reinterpret_cast<uint4*>(o_hi + tok * kC + head * kHd + c * 8) = val;
        } else if (FMT == FMT_SPLIT16) {
          *reinterpret_cast<uint4*>(o_lo + tok * kC + head * kHd + (c - 8) * 8) = val;
        } else {      // c8 row = 1024 B: [0,512) e5m2(x 2^-8), [512,1024) e5m2(lo 2^4); this head owns 64 B of each
          uint8_t* c8 = reinterpret_cast<uint8_t*>(o_lo) + tok * (2 * kC) + head * kHd;
          *reinterpret_cast<uint4*>(c8 + (c < 12 ? 0 : kC) + ((c - 8) & 3) * 16) = val;
        }
      }
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------ spatial, J = 17
constexpr int SJ = 17;
constexpr int kSpRows = 3 * SJ + 1;                 // q, k, v tiles of one head + one all-zero row
constexpr int kSpWarpHalves = kSpRows * KS;         // 3744 halves = 7488 B per warp

template <int FMT>
__global__ void __launch_bounds__(256, 3)
attn_spatial_h16_kernel(const __half* __restrict__ qkv, __half* __restrict__ o_hi, __half* __restrict__ o_lo,
                        float* __restrict__ o_f32, int64_t n_groups) {
  extern __shared__ __align__(16) __half smh[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int head = warp;                                    // 8 warps = 8 heads of one frame
  const int64_t grp = blockIdx.x;
  if (grp >= n_groups) return;
  __half* Qs = smh + warp * kSpWarpHalves;
  __half* Ksm = Qs + SJ * KS;
  __half* Vsm = Ksm + SJ * KS;
  const uint32_t sQ = static_cast<uint32_t>(__cvta_generic_to_shared(Qs));
  const uint32_t sK = sQ + SJ * KS * 2, sV = sK + SJ * KS * 2, sZ = sV + SJ * KS * 2;
  const __half* base = qkv + static_cast<size_t>(grp) * SJ * kQkvRow + head * kHd;

  // ---- q, k, v_hi rows of this head: 17 x 3 x 128 B, 16 B per cp.async
  for (int i = lane; i < 3 * SJ * 8; i += 32) {
    const int c8 = i & 7, rw = i >> 3;                      // rw = which * 17 + token
    const int which = rw / SJ, tokn = rw - which * SJ;
    cp_async16(sQ + static_cast<uint32_t>((rw * KS + c8 * 8) * 2),
               base + static_cast<size_t>(tokn) * kQkvRow + which * kC + c8 * 8);
  }
  if (lane < 9) asm volatile("st.shared.v4.u32 [%0], {%1,%1,%1,%1};" ::"r"(sZ + lane * 16), "r"(0u) : "memory");
  cp_async_wait_all();
  __syncwarp();

  const int g = lane >> 2, q4 = lane & 3;
  // ldmatrix row providers (row index within a 16-row group) and column offsets
  const int a_row = (lane & 7) + (((lane >> 3) & 1) << 3), a_col = (lane >> 4) << 3;       // A operand (Q)
  const int k_key = (lane & 7) + ((lane >> 4) << 3), k_d = ((lane >> 3) & 1) << 3;         // B operand (K)
  const int v_key = a_row, v_d = a_col;                                                    // B operand (V, .trans)
  auto row_addr = [&](uint32_t tile, int row, int col) -> uint32_t {       // rows >= 17 read the zero row
    return row < SJ ? tile + static_cast<uint32_t>((row * KS + col) * 2) : sZ + static_cast<uint32_t>((col & 63) * 2);
  };

  // One 16-query m-tile: S = Q K^T (3 key n-tiles), softmax over the 17 real keys, O = P V / l.
  auto tile = [&](int mt, float (&o)[8][4]) {
    float s[3][4];
#pragma unroll
    for (int i = 0; i < 3; ++i) { s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f; }
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      uint32_t a[4], b01[4], b2[4];
      ldsm_x4(row_addr(sQ, mt * 16 + a_row, ks * 16 + a_col), a);
      ldsm_x4(row_addr(sK, k_key, ks * 16 + k_d), b01);               // keys 0..15
      ldsm_x4(row_addr(sK, 16 + k_key, ks * 16 + k_d), b2);           // keys 16..31 (only 16 is real)
      mma16816(s[0], a, b01[0], b01[1]);
      mma16816(s[1], a, b01[2], b01[3]);
      mma16816(s[2], a, b2[0], b2[1]);
    }
    // softmax in the exp2 domain; rows g and g+8 of this m-tile
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < 3; ++nt) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int key = nt * 8 + 2 * q4 + (e & 1);
        const float v = key < SJ ? s[nt][e] * kScaleLog2e : -INFINITY;
        s[nt][e] = v;
        if (e < 2) mx0 = fmaxf(mx0, v); else mx1 = fmaxf(mx1, v);
      }
    }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    float l0 = 0.f, l1 = 0.f;
#pragma unroll
    for (int nt = 0; nt < 3; ++nt) {
      s[nt][0] = ex2_approx(s[nt][0] - mx0); s[nt][1] = ex2_approx(s[nt][1] - mx0);
      s[nt][2] = ex2_approx(s[nt][2] - mx1); s[nt][3] = ex2_approx(s[nt][3] - mx1);
      l0 += s[nt][0] + s[nt][1];
      l1 += s[nt][2] + s[nt][3];
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float i0 = rcp_approx(l0), i1 = rcp_approx(l1);
    // O = P V: k-step 0 = keys 0..15, k-step 1 = keys 16..31 (P is zero beyond key 16)
    uint32_t pa0[4], pa1[4];
    pa0[0] = pack2f(s[0][0], s[0][1]); pa0[1] = pack2f(s[0][2], s[0][3]);
    pa0[2] = pack2f(s[1][0], s[1][1]); pa0[3] = pack2f(s[1][2], s[1][3]);
    pa1[0] = pack2f(s[2][0], s[2][1]); pa1[1] = pack2f(s[2][2], s[2][3]);
    pa1[2] = 0u; pa1[3] = 0u;
#pragma unroll
    for (int i = 0; i < 8; ++i) { o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f; }
#pragma unroll
    for (int dp = 0; dp < 4; ++dp) {
      uint32_t v0[4], v1[4];
      ldsm_x4_t(row_addr(sV, v_key, dp * 16 + v_d), v0);
      ldsm_x4_t(row_addr(sV, 16 + v_key, dp * 16 + v_d), v1);
      mma16816(o[2 * dp], pa0, v0[0], v0[1]);
      mma16816(o[2 * dp + 1], pa0, v0[2], v0[3]);
      mma16816(o[2 * dp], pa1, v1[0], v1[1]);
      mma16816(o[2 * dp + 1], pa1, v1[2], v1[3]);
    }
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) { o[nt][0] *= i0; o[nt][1] *= i0; o[nt][2] *= i1; o[nt][3] *= i1; }
  };

  // m-tile 1 first: of its 16 rows only joint 16 is real (row g == 0, first half) -> keep 16 values
  float o16[8][2];
  {
    float o[8][4];
    tile(1, o);
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) { o16[nt][0] = o[nt][0]; o16[nt][1] = o[nt][1]; }
  }
  float o0[8][4];
  tile(0, o0);
  __syncwarp();        // every lane is done reading Q / K through ldmatrix: their tiles become the output stage

  // ---- out = P V / l - (v_hi + v_lo); staged per row in shared memory (hi -> Q tile, lo -> K tile; fp32 uses both)
  const __half* vlo_base = base + 3 * kC;
  auto stage_row = [&](int r, const float (&x)[8][2]) {     // x[nt] = columns nt*8 + 2*q4, +1 of row r (P V / l)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const int d = nt * 8 + 2 * q4;
      const __half2 vh = *reinterpret_cast<const __half2*>(Vsm + r * KS + d);
      const __half2 vl = __ldg(reinterpret_cast<const __half2*>(vlo_base + static_cast<size_t>(r) * kQkvRow + d));
      const float x0 = x[nt][0] - (__low2float(vh) + __low2float(vl));
      const float x1 = x[nt][1] - (__high2float(vh) + __high2float(vl));
      if (o_f32) {          // fp32 row = 256 B: first 32 floats in the Q tile row, last 32 in the K tile row
        float* dstrow = reinterpret_cast<float*>((d < 32 ? Qs : Ksm) + r * KS);
        *reinterpret_cast<float2*>(dstrow + (d & 31)) = make_float2(x0, x1);
      } else if (FMT == FMT_SPLIT16) {
        uint32_t hh, ll;
        split2(x0, x1, hh, ll);
        *reinterpret_cast<uint32_t*>(Qs + r * KS + d) = hh;
        *reinterpret_cast<uint32_t*>(Ksm + r * KS + d) = ll;
      } else {              // K tile row: e5m2(x 2^-8) in bytes [0,64), e5m2(lo 2^4) in bytes [64,128)
        const __half h0 = __float2half_rn(x0), h1 = __float2half_rn(x1);
        *reinterpret_cast<uint32_t*>(Qs + r * KS + d) = pack2(h0, h1);
        uint8_t* krow = reinterpret_cast<uint8_t*>(Ksm + r * KS);
        *reinterpret_cast<uint16_t*>(krow + d) = static_cast<uint16_t>(op_e5m2x2(x0 * kActHiScale, x1 * kActHiScale));
        *reinterpret_cast<uint16_t*>(krow + 64 + d) = static_cast<uint16_t>(
            op_e5m2x2((x0 - __half2float(h0)) * kActLoScale, (x1 - __half2float(h1)) * kActLoScale));
      }
    }
  };
  {
    float x[8][2];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) { x[nt][0] = o0[nt][0]; x[nt][1] = o0[nt][1]; }
    stage_row(g, x);
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) { x[nt][0] = o0[nt][2]; x[nt][1] = o0[nt][3]; }
    stage_row(g + 8, x);
    if (g == 0) stage_row(16, o16);
  }
  __syncwarp();
  const size_t tok_base = static_cast<size_t>(grp) * SJ;
  if (o_f32) {
    for (int i = lane; i < SJ * 16; i += 32) {            // 16 x 16 B per row
      const int r = i >> 4, c = i & 15;
      const uint4 v = *reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>((c < 8 ? Qs : Ksm) + r * KS) + (c & 7) * 16);
      *reinterpret_cast<uint4*>(o_f32 + (tok_base + r) * kC + head * kHd + c * 4) = v;
    }
  } else {
    for (int i = lane; i < SJ * 16; i += 32) {            // 8 x 16 B of hi and 8 x 16 B of lo per row
      const int r = i >> 4, c = i & 15;
      const uint4 v = *reinterpret_cast<const uint4*>((c < 8 ? Qs : Ksm) + r * KS + (c & 7) * 8);
      if (c < 8 || FMT == FMT_SPLIT16) {
        __half* dst = (c < 8 ? o_hi : o_lo) + (tok_base + r) * kC + head * kHd + (c & 7) * 8;
        *reinterpret_cast<uint4*>(dst) = v;
      } else {
        uint8_t* c8 = reinterpret_cast<uint8_t*>(o_lo) + (tok_base + r) * (2 * kC) + head * kHd;
        *reinterpret_cast<uint4*>(c8 + (c < 12 ? 0 : kC) + ((c - 8) & 3) * 16) = v;
      }
    }
  }
}

constexpr int kSpatialSmem = 8 * kSpWarpHalves * static_cast<int>(sizeof(__half));   // 59904 B

}  // namespace

cudaError_t configure_attention_mma() {
  const int tsmem = 2 * 256 * KS * static_cast<int>(sizeof(__half)) + 8 * kTStgWarp;
  cudaError_t e;
  if ((e = cudaFuncSetAttribute(attn_temporal_h16_kernel<FMT_SPLIT16>, cudaFuncAttributeMaxDynamicSharedMemorySize, tsmem)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(attn_temporal_h16_kernel<FMT_F8C>, cudaFuncAttributeMaxDynamicSharedMemorySize, tsmem)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(attn_spatial_h16_kernel<FMT_SPLIT16>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSpatialSmem)) != cudaSuccess) return e;
  return cudaFuncSetAttribute(attn_spatial_h16_kernel<FMT_F8C>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSpatialSmem);
}

cudaError_t launch_attn_temporal_mma(const __half* qkv, __half* o_hi, __half* o_lo, float* o_f32, int fmt, int B, int F,
                                     int J, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  if (F < 1 || F > 256) return cudaErrorInvalidValue;
  const int NK = (F + 63) / 64 * 64;
  const int n_qt = (F + 15) / 16;
  const int warps = n_qt < 8 ? n_qt : 8;
  const int smem = 2 * NK * KS * static_cast<int>(sizeof(__half)) + warps * kTStgWarp;
  dim3 grid(static_cast<unsigned>(B) * J, kHeads);
  auto kern = fmt == FMT_F8C ? attn_temporal_h16_kernel<FMT_F8C> : attn_temporal_h16_kernel<FMT_SPLIT16>;
  kern<<<grid, warps * 32, smem, st>>>(qkv, o_hi, o_lo, o_f32, F, J, NK);
  return cudaGetLastError();
}

cudaError_t launch_attn_spatial(const __half* qkv, __half* o_hi, __half* o_lo, float* o_f32, int fmt, int64_t n_groups,
                                int J, cudaStream_t st) {
  if (n_groups <= 0) return cudaSuccess;
  if (J != SJ) return cudaErrorInvalidValue;
  auto kern = fmt == FMT_F8C ? attn_spatial_h16_kernel<FMT_F8C> : attn_spatial_h16_kernel<FMT_SPLIT16>;
  kern<<<static_cast<unsigned>(n_groups), 256, kSpatialSmem, st>>>(qkv, o_hi, o_lo, o_f32, n_groups);
  return cudaGetLastError();
}

}  // namespace d3d
