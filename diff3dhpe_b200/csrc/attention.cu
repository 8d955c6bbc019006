// CUDA-core (fp32 arithmetic) GRAND attention used ONLY to validate the tensor-core kernels of attention_mma.cu:
// same packed fp16 input (row = q | k | v_hi | v_lo, see EPI_QKV16), same output formats, no tensor cores.
//
//     O = (softmax(Q K^T * hd^-0.5) - I) V        (MODEL:76-83)
//
// One CTA per (sequence, head).  Token of position n in sequence s:  (s / inner) * outer + (s % inner) + n * tok_stride
//   spatial : inner = 1, outer = J, tok_stride = 1, N = J      (s = b*F + f)
//   temporal: inner = J, outer = F*J, tok_stride = J, N = F    (s = b*J + j)   -- no transposes (MODEL:119-121,130-133)
// Also: pack_qkv16_kernel, fp32 [T, 3 C] -> the packed fp16 layout (op-level test entry point only; in the
// sampler the qkv GEMM epilogue writes the packed layout directly).  The validation kernel is built for C = 512 only.
#include "kernels.cuh"
#include "operand.cuh"

namespace d3d {
namespace {

constexpr int kC = Width<512>::kC, kHd = Width<512>::kHd, kQkvRow = Width<512>::kQkvRow;
constexpr float kScale = 0.125f;   // head_dim ** -0.5, MODEL:65
constexpr int KPAD = kHd + 1;

__device__ __forceinline__ uint32_t pack2(__half a, __half b) {
  return static_cast<uint32_t>(__half_as_ushort(a)) | (static_cast<uint32_t>(__half_as_ushort(b)) << 16);
}

__global__ void __launch_bounds__(256)
attn_generic_kernel(const __half* __restrict__ qkv, __half* __restrict__ o_hi, __half* __restrict__ o_lo,
                    float* __restrict__ o_f32, int fmt, int N, int64_t outer, int inner, int64_t tok_stride) {
  extern __shared__ float sm[];
  float* Ks = sm;                       // [N][65]
  float* Vs = Ks + ((N * KPAD + 3) & ~3);   // [N][64], 16-byte aligned
  float* Ps = Vs + N * kHd;             // [8][N]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int head = blockIdx.y;
  const int64_t s = blockIdx.x;
  const int64_t tok0 = (s / inner) * outer + (s % inner);
  const __half* base = qkv + head * kHd;

  for (int i = threadIdx.x; i < N * kHd; i += blockDim.x) {
    const int r = i >> 6, d = i & 63;
    const size_t row = static_cast<size_t>(tok0 + r * tok_stride) * kQkvRow;
    Ks[r * KPAD + d] = __half2float(base[row + kC + d]);
    Vs[r * kHd + d] = __half2float(base[row + 2 * kC + d]) + __half2float(base[row + 3 * kC + d]);
  }
  __syncthreads();

  float* P = Ps + warp * N;
  for (int i = warp; i < N; i += 8) {
    float q[kHd];
    const __half* qrow = base + static_cast<size_t>(tok0 + i * tok_stride) * kQkvRow;
#pragma unroll
    for (int d = 0; d < kHd; ++d) q[d] = __half2float(qrow[d]);
    float sc[8];
    float mx = -INFINITY;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int kk = lane + 32 * it;
      float a = -INFINITY;
      if (kk < N) {
        a = 0.f;
        const float* kr = Ks + kk * KPAD;
#pragma unroll
        for (int d = 0; d < kHd; ++d) a = fmaf(q[d], kr[d], a);
        a *= kScale;
      }
      sc[it] = a;
      mx = fmaxf(mx, a);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int kk = lane + 32 * it;
      sc[it] = kk < N ? expf(sc[it] - mx) : 0.f;
      sum += sc[it];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float inv = 1.0f / sum;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int kk = lane + 32 * it;
      if (kk < N) P[kk] = sc[it] * inv - (kk == i ? 1.0f : 0.0f);
    }
    __syncwarp();
    float o0 = 0.f, o1 = 0.f;
    for (int kk = 0; kk < N; ++kk) {
      const float p = P[kk];
      const float2 vv = *reinterpret_cast<const float2*>(Vs + kk * kHd + 2 * lane);
      o0 = fmaf(p, vv.x, o0);
      o1 = fmaf(p, vv.y, o1);
    }
    __syncwarp();
    const size_t off = static_cast<size_t>(tok0 + i * tok_stride) * kC + head * kHd + 2 * lane;
    if (o_f32) {
      *reinterpret_cast<float2*>(o_f32 + off) = make_float2(o0, o1);
    } else {
      const __half h0 = __float2half_rn(o0), h1 = __float2half_rn(o1);
      *reinterpret_cast<uint32_t*>(o_hi + off) = pack2(h0, h1);
      if (fmt == FMT_SPLIT16) {
        *reinterpret_cast<uint32_t*>(o_lo + off) =
            pack2(__float2half_rn(o0 - __half2float(h0)), __float2half_rn(o1 - __half2float(h1)));
      } else {
        uint8_t* c8 = reinterpret_cast<uint8_t*>(o_lo) + static_cast<size_t>(tok0 + i * tok_stride) * (2 * kC) +
                      head * kHd + 2 * lane;
        *reinterpret_cast<uint16_t*>(c8) = static_cast<uint16_t>(op_e5m2x2(o0 * kActHiScale, o1 * kActHiScale));
        *reinterpret_cast<uint16_t*>(c8 + kC) = static_cast<uint16_t>(
            op_e5m2x2((o0 - __half2float(h0)) * kActLoScale, (o1 - __half2float(h1)) * kActLoScale));
      }
    }
  }
}

template <int C>
__global__ void pack_qkv16_kernel(const float* __restrict__ in, __half* __restrict__ out, int64_t T) {
  constexpr int kRow = Width<C>::kQkvRow;
  const int64_t n = T * (3 * C);
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t t = i / (3 * C);
    const int c = static_cast<int>(i - t * (3 * C));
    const float v = in[i];
    const __half h = __float2half_rn(v);
    out[t * kRow + c] = h;
    if (c >= 2 * C) out[t * kRow + c + C] = __float2half_rn(v - __half2float(h));
  }
}

}  // namespace

cudaError_t configure_attention() {
  return cudaFuncSetAttribute(attn_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              (((256 * KPAD + 3) & ~3) + 256 * kHd + 8 * 256) * static_cast<int>(sizeof(float)));
}

cudaError_t launch_attn_generic_simt(const __half* qkv, __half* o_hi, __half* o_lo, float* o_f32, int fmt, int n_seq,
                                     int N, int64_t outer, int inner, int64_t tok_stride, cudaStream_t st) {
  if (n_seq <= 0) return cudaSuccess;
  if (N < 1 || N > 256) return cudaErrorInvalidValue;
  const int smem = (((N * KPAD + 3) & ~3) + N * kHd + 8 * N) * static_cast<int>(sizeof(float));
  dim3 grid(static_cast<unsigned>(n_seq), kHeads);
  attn_generic_kernel<<<grid, 256, smem, st>>>(qkv, o_hi, o_lo, o_f32, fmt, N, outer, inner, tok_stride);
  return cudaGetLastError();
}

cudaError_t launch_attn_temporal_simt(const __half* qkv, __half* o_hi, __half* o_lo, float* o_f32, int fmt, int B, int F,
                                      int J, cudaStream_t st) {
  return launch_attn_generic_simt(qkv, o_hi, o_lo, o_f32, fmt, B * J, F, static_cast<int64_t>(F) * J, J, J, st);
}

cudaError_t launch_pack_qkv16(int C, const float* qkv_f32, __half* out, int64_t T, cudaStream_t st) {
  if (T <= 0) return cudaSuccess;
  if (!width_supported(C)) return cudaErrorInvalidValue;
  int64_t g = (T * 3 * C + 255) / 256;
  if (g > 148 * 32) g = 148 * 32;
  if (C == 256) pack_qkv16_kernel<256><<<static_cast<unsigned>(g), 256, 0, st>>>(qkv_f32, out, T);
  else pack_qkv16_kernel<512><<<static_cast<unsigned>(g), 256, 0, st>>>(qkv_f32, out, T);
  return cudaGetLastError();
}

}  // namespace d3d
