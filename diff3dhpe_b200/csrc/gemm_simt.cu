// CUDA-core fp32 validation GEMM.  Consumes exactly the operands of the tcgen05 kernel (fp16 hi/lo halves,
// K-major) and produces exactly its outputs, so the tensor-core path can be checked element by element on
// the device.  Not a performance path: 64x64 tiles, 4x4 outputs per thread.
#include "kernels.cuh"
#include "operand.cuh"

namespace d3d {
namespace {

// CUDA-core validation GEMM: its packed q|k|v epilogue is built for C = 512 only
constexpr int kC = Width<512>::kC, kQkvRow = Width<512>::kQkvRow;

constexpr int TM = 64, TN = 64, TK = 16;

__device__ __forceinline__ float gelu_erf(float v) { return 0.5f * v * (1.0f + erff(v * 0.70710678118654752440f)); }

// FMT_SPLIT16: acc = (a_hi + a_lo) . (b_hi + b_lo)   (the lo.lo term, 2^-22 relative, is the only difference from the
//              3-pass tensor-core kernel).
// FMT_F8C    : acc = a_hi . b_hi + a8 . blo8 + alo8 . b8 with the e5m2 factors decoded to fp32: exactly the products the
//              tensor-core kernel forms (the power-of-two scales cancel), so it validates that kernel tightly.
// FMT_F4C    : the same with the correction factors decoded from block-scaled e2m1 (nibble x 2^(scale byte - 127)):
//              exactly what tcgen05.mma kind::mxf4.block_scale multiplies.
// value of element k of part `part` (0 = P, 1 = Q) of row `row` of a FMT_F4C operand with inner dimension K
__device__ __forceinline__ float f4c_value(const uint8_t* __restrict__ c4, const uint8_t* __restrict__ sf, int64_t row,
                                           int k, int part, int K) {
  const uint32_t byte = c4[row * K + part * (K >> 1) + (k >> 1)];
  const float q = op_e2m1_to_float((k & 1) ? (byte >> 4) : (byte & 15u));
  return q * op_ue8m0_val(sf[op_sf_offset(row, part * (K >> 5) + (k >> 5), K / 64)]);
}

template <int EPI, int FMT>
__global__ void __launch_bounds__(256)
gemm_simt_kernel(const __half* __restrict__ a_hi, const __half* __restrict__ a_lo, const uint8_t* __restrict__ a_sf,
                 const __half* __restrict__ b_hi, const __half* __restrict__ b_lo, const uint8_t* __restrict__ b_sf,
                 const __grid_constant__ GemmParams p) {
  __shared__ float As[TK][TM + 1];
  __shared__ float Bs[TK][TN + 1];
  __shared__ float A8[FMT != FMT_SPLIT16 ? 2 * TK : 1][TM + 1];  // F8C: [0,TK) e5m2(a 2^-8), [TK,2TK) e5m2(a_lo 2^4); F4C: P, Q
  __shared__ float B8[FMT != FMT_SPLIT16 ? 2 * TK : 1][TN + 1];  // F8C: [0,TK) e5m2(b_lo 2^8), [TK,2TK) e5m2(b 2^-4); F4C: P, Q
  const uint8_t* a_c8 = reinterpret_cast<const uint8_t*>(a_lo);
  const uint8_t* b_c8 = reinterpret_cast<const uint8_t*>(b_lo);
  const int m0 = blockIdx.x * TM, n0 = blockIdx.y * TN;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < p.K; k0 += TK) {
    for (int i = threadIdx.x; i < TM * TK; i += 256) {
      const int r = i / TK, c = i % TK;
      const int gm = m0 + r;
      float v = 0.f, v8 = 0.f, vl8 = 0.f;
      if (gm < p.M) {
        const size_t o = static_cast<size_t>(gm) * p.K + k0 + c;
        v = __half2float(a_hi[o]);
        if (FMT == FMT_SPLIT16) {
          if (a_lo) v += __half2float(a_lo[o]);
        } else if (FMT == FMT_F4C) {
          v8 = f4c_value(a_c8, a_sf, gm, k0 + c, 0, p.K);
          vl8 = f4c_value(a_c8, a_sf, gm, k0 + c, 1, p.K);
        } else {
          const size_t o8 = static_cast<size_t>(gm) * 2 * p.K + k0 + c;
          v8 = op_e5m2_to_float(a_c8[o8]);
          vl8 = op_e5m2_to_float(a_c8[o8 + p.K]);
        }
      }
      As[c][r] = v;
      const size_t ob = static_cast<size_t>(n0 + r) * p.K + k0 + c;
      float w = __half2float(b_hi[ob]);
      if (FMT == FMT_SPLIT16) {
        if (b_lo) w += __half2float(b_lo[ob]);
      } else if (FMT == FMT_F4C) {
        A8[c][r] = v8; A8[TK + c][r] = vl8;
        B8[c][r] = f4c_value(b_c8, b_sf, n0 + r, k0 + c, 0, p.K);
        B8[TK + c][r] = f4c_value(b_c8, b_sf, n0 + r, k0 + c, 1, p.K);
      } else {
        const size_t ob8 = static_cast<size_t>(n0 + r) * 2 * p.K + k0 + c;
        A8[c][r] = v8; A8[TK + c][r] = vl8;
        B8[c][r] = op_e5m2_to_float(b_c8[ob8]); B8[TK + c][r] = op_e5m2_to_float(b_c8[ob8 + p.K]);
      }
      Bs[c][r] = w;
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < TK; ++k) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[k][ty * 4 + i]; b[i] = Bs[k][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (FMT != FMT_SPLIT16) {
#pragma unroll 8
      for (int k = 0; k < 2 * TK; ++k) {
        float a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { a[i] = A8[k][ty * 4 + i]; b[i] = B8[k][tx * 4 + i]; }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
    }
    __syncthreads();
  }
  if (EPI == EPI_GELU_SPLIT && FMT == FMT_F4C) {
    // block-scaled output operand: a 32-column scale block = the 4 columns of 8 consecutive tx (lanes tx & ~7 .. | 7)
    uint8_t* c4 = reinterpret_cast<uint8_t*>(p.out_lo);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int gm = m0 + ty * 4 + i;
      const int gn = n0 + tx * 4;
      float x[4], l[4];
      __half hh[4];
      float ax = 0.f, al = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        x[j] = gelu_erf(acc[i][j] + p.bias[gn + j]);
        hh[j] = __float2half_rn(x[j]);
        l[j] = x[j] - __half2float(hh[j]);
        ax = fmaxf(ax, fabsf(x[j]));
        al = fmaxf(al, fabsf(l[j]));
      }
#pragma unroll
      for (int o = 1; o < 8; o <<= 1) {
        ax = fmaxf(ax, __shfl_xor_sync(0xffffffffu, ax, o));
        al = fmaxf(al, __shfl_xor_sync(0xffffffffu, al, o));
      }
      if (gm >= p.M) continue;
      const uint32_t bp = op_ue8m0_of(ax), bq = op_ue8m0_of(al);
      const float ip = op_ue8m0_inv(bp), iq = op_ue8m0_inv(bq);
#pragma unroll
      for (int j = 0; j < 4; ++j) p.out_hi[static_cast<size_t>(gm) * p.N + gn + j] = hh[j];
      uint8_t* crow = c4 + static_cast<size_t>(gm) * p.N;
      *reinterpret_cast<uint16_t*>(crow + (gn >> 1)) =
          static_cast<uint16_t>(op_e2m1x2(x[0] * ip, x[1] * ip) | (op_e2m1x2(x[2] * ip, x[3] * ip) << 8));
      *reinterpret_cast<uint16_t*>(crow + (p.N >> 1) + (gn >> 1)) =
          static_cast<uint16_t>(op_e2m1x2(l[0] * iq, l[1] * iq) | (op_e2m1x2(l[2] * iq, l[3] * iq) << 8));
      if ((tx & 7) == 0) {
        p.out_sf[op_sf_offset(gm, gn >> 5, p.N / 64)] = static_cast<uint8_t>(bp);
        p.out_sf[op_sf_offset(gm, (p.N >> 5) + (gn >> 5), p.N / 64)] = static_cast<uint8_t>(bq);
      }
    }
    return;
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gm = m0 + ty * 4 + i;
    if (gm >= p.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gn = n0 + tx * 4 + j;
      const size_t o = static_cast<size_t>(gm) * p.N + gn;
      float v = acc[i][j] + p.bias[gn];
      if (EPI == EPI_F32) {
        if (p.residual) v += p.residual[o];
        p.out_f32[o] = v;
      } else if (EPI == EPI_GELU_SPLIT) {
        v = gelu_erf(v);
        const __half h = __float2half_rn(v);
        p.out_hi[o] = h;
        if (FMT == FMT_SPLIT16) {
          p.out_lo[o] = __float2half_rn(v - __half2float(h));
        } else {
          uint8_t* c8 = reinterpret_cast<uint8_t*>(p.out_lo) + static_cast<size_t>(gm) * 2 * p.N + gn;
          c8[0] = static_cast<uint8_t>(op_e5m2x2(v * kActHiScale, 0.f) & 0xff);
          c8[p.N] = static_cast<uint8_t>(op_e5m2x2((v - __half2float(h)) * kActLoScale, 0.f) & 0xff);
        }
      } else {   // EPI_QKV16
        const size_t oq = static_cast<size_t>(gm) * kQkvRow + gn;
        const __half h = __float2half_rn(v);
        p.out_qkv[oq] = h;
        if (gn >= 2 * kC) p.out_qkv[oq + kC] = __float2half_rn(v - __half2float(h));
      }
    }
  }
}

}  // namespace

cudaError_t launch_gemm_simt(const __half* a_hi, const __half* a_lo, const uint8_t* a_sf, const __half* b_hi,
                             const __half* b_lo, const uint8_t* b_sf, const GemmParams& p, int epi, int fmt,
                             cudaStream_t st) {
  if (p.M <= 0) return cudaSuccess;
  if (p.N % TN != 0 || p.K % TK != 0) return cudaErrorInvalidValue;
  if (fmt == FMT_F4C && (p.K % 64 != 0 || !a_sf || !b_sf || (epi == EPI_GELU_SPLIT && !p.out_sf))) return cudaErrorInvalidValue;
  dim3 grid((p.M + TM - 1) / TM, p.N / TN);
#define D3D_SIMT(EPI_, FMT_) gemm_simt_kernel<EPI_, FMT_><<<grid, 256, 0, st>>>(a_hi, a_lo, a_sf, b_hi, b_lo, b_sf, p)
  if (fmt == FMT_F4C) {
    if (epi == EPI_F32) D3D_SIMT(EPI_F32, FMT_F4C);
    else if (epi == EPI_GELU_SPLIT) D3D_SIMT(EPI_GELU_SPLIT, FMT_F4C);
    else D3D_SIMT(EPI_QKV16, FMT_F4C);
  } else if (fmt == FMT_F8C) {
    if (epi == EPI_F32) D3D_SIMT(EPI_F32, FMT_F8C);
    else if (epi == EPI_GELU_SPLIT) D3D_SIMT(EPI_GELU_SPLIT, FMT_F8C);
    else D3D_SIMT(EPI_QKV16, FMT_F8C);
  } else {
    if (epi == EPI_F32) D3D_SIMT(EPI_F32, FMT_SPLIT16);
    else if (epi == EPI_GELU_SPLIT) D3D_SIMT(EPI_GELU_SPLIT, FMT_SPLIT16);
    else D3D_SIMT(EPI_QKV16, FMT_SPLIT16);
  }
#undef D3D_SIMT
  return cudaGetLastError();
}

}  // namespace d3d
