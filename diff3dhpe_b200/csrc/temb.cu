// G-temb: sinusoidal time embedding and the tiny time MLPs (MODEL:29-36, 169-174, 104-116).
// At eval every clip of a DDIM step shares one t (DIFF:254), so the whole [S, 2*depth, C] table of
// per-block time vectors is computed once per (weights, schedule); the same kernels serve the general
// per-sample-t path of forward_denoise.  Work is O(R * 10 MFLOP): fp32 CUDA cores, one warp per output.
#include "kernels.cuh"

namespace d3d {
namespace {

template <int C>
__global__ void sincos_kernel(const float* __restrict__ t, int R, float* __restrict__ out) {
  constexpr int kHalf = C / 2;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;      // over R * C / 2
  if (i >= R * kHalf) return;
  const int r = i / kHalf, k = i % kHalf;
  // freq_k = exp(k * -(ln(1e4)/(half_dim - 1))) evaluated like torch does in fp32: the product k * (-step) is rounded to
  // fp32, exp is correctly rounded from double; arg = t * freq in fp32; sin/cos correctly rounded from double.
  const float step = static_cast<float>(9.210340371976184 / (kHalf - 1.0));   // math.log(10000) / (half_dim - 1)
  const float e = __fmul_rn(static_cast<float>(k), -step);
  const float freq = static_cast<float>(exp(static_cast<double>(e)));
  const float arg = __fmul_rn(t[r], freq);
  out[r * C + k] = static_cast<float>(sin(static_cast<double>(arg)));
  out[r * C + kHalf + k] = static_cast<float>(cos(static_cast<double>(arg)));
}

// per-sample timesteps of forward_denoise (int64 on the device, MODEL:33 multiplies them into fp32) -> fp32
__global__ void t_to_f32_kernel(const int64_t* __restrict__ t, int R, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < R) out[i] = static_cast<float>(t[i]);
}

__device__ __forceinline__ float act(float v, int mode) {
  if (mode == 1) return 0.5f * v * (1.0f + erff(v * 0.70710678118654752440f));   // nn.GELU (erf)
  if (mode == 2) return v / (1.0f + expf(-v));                                   // nn.SiLU
  return v;
}

__global__ void __launch_bounds__(256)
small_linear_kernel(const float* __restrict__ in, int R, int K, const float* __restrict__ W,
                    const float* __restrict__ b, int N, int act_in, float* __restrict__ out, int64_t out_row_stride) {
  const int lane = threadIdx.x & 31;
  const int64_t w = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (w >= static_cast<int64_t>(R) * N) return;
  const int r = static_cast<int>(w / N), n = static_cast<int>(w % N);
  const float* x = in + static_cast<size_t>(r) * K;
  const float* wr = W + static_cast<size_t>(n) * K;
  float a = 0.f;
  for (int k = 4 * lane; k < K; k += 128) {
    const float4 xv = *reinterpret_cast<const float4*>(x + k);
    const float4 wv = __ldg(reinterpret_cast<const float4*>(wr + k));
    a = fmaf(act(xv.x, act_in), wv.x, a);
    a = fmaf(act(xv.y, act_in), wv.y, a);
    a = fmaf(act(xv.z, act_in), wv.z, a);
    a = fmaf(act(xv.w, act_in), wv.w, a);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  if (lane == 0) out[static_cast<size_t>(r) * out_row_stride + n] = a + b[n];
}

}  // namespace

cudaError_t launch_t_to_f32(const int64_t* t, int R, float* out, cudaStream_t st) {
  if (R <= 0) return cudaSuccess;
  t_to_f32_kernel<<<(R + 255) / 256, 256, 0, st>>>(t, R, out);
  return cudaGetLastError();
}

cudaError_t launch_sincos(int C, const float* t, int R, float* out, cudaStream_t st) {
  if (R <= 0) return cudaSuccess;
  if (!width_supported(C)) return cudaErrorInvalidValue;
  if (C == 256) sincos_kernel<256><<<(R * 128 + 255) / 256, 256, 0, st>>>(t, R, out);
  else sincos_kernel<512><<<(R * 256 + 255) / 256, 256, 0, st>>>(t, R, out);
  return cudaGetLastError();
}

cudaError_t launch_small_linear(const float* in, int R, int K, const float* W, const float* b, int N, int act_in,
                                float* out, int64_t out_row_stride, cudaStream_t st) {
  if (R <= 0) return cudaSuccess;
  if (K % 4 != 0) return cudaErrorInvalidValue;
  const int64_t warps = static_cast<int64_t>(R) * N;
  small_linear_kernel<<<static_cast<unsigned>((warps + 7) / 8), 256, 0, st>>>(in, R, K, W, b, N, act_in, out,
                                                                              out_row_stride);
  return cudaGetLastError();
}

}  // namespace d3d
