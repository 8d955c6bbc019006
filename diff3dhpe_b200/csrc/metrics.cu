// Protocol #1 / #2 / #3 errors and the velocity error of evaluate() on the device (SURVEY.md 8f N4):
//   mpjpe (LOSS:15-27), n_mpjpe (LOSS:84-94), p_mpjpe (LOSS:43-82: Procrustes alignment, numpy SVD on the host in the
//   reference) and mean_velocity_error (LOSS:133-142), accumulated as fp64 sums so that the whole tail of RUN:602-614
//   stays on the GPU.  LOSS = common/loss.py.  One thread per frame; the 3 x 3 SVD is a cyclic Jacobi
//   eigen-decomposition of H^T H in fp64.
// Also the per-joint error histogram behind the MPI-INF-3DHP PCK / AUC table (pck_hist_kernel).
#include "kernels.cuh"

namespace d3d {
namespace {

constexpr int kMaxJ = 32;

__device__ __forceinline__ void jacobi_rotate(double (&a)[3][3], double (&v)[3][3], int p, int q) {
  if (fabs(a[p][q]) < 1e-300) return;
  const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
  const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
  const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
#pragma unroll
  for (int k = 0; k < 3; ++k) {            // A <- A G
    const double akp = a[k][p], akq = a[k][q];
    a[k][p] = c * akp - s * akq;
    a[k][q] = s * akp + c * akq;
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {            // A <- G^T A
    const double apk = a[p][k], aqk = a[q][k];
    a[p][k] = c * apk - s * aqk;
    a[q][k] = s * apk + c * aqk;
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {            // V <- V G
    const double vkp = v[k][p], vkq = v[k][q];
    v[k][p] = c * vkp - s * vkq;
    v[k][q] = s * vkp + c * vkq;
  }
}

// acc[0] += sum_j |p - g|, acc[1] += sum_j |s p - g| (n_mpjpe), acc[2] += sum_j |aligned(p) - g| (p_mpjpe),
// acc[3] += joints counted; vel_tmp[0] += sum of velocity-error norms over consecutive SELECTED frames, vel_tmp[1] +=
// their count (this call only; vel_finalize_kernel folds them into acc[4], acc[5])
__global__ void pose_metrics_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                    const int64_t* __restrict__ sel, int64_t n_sel, int J, double* __restrict__ acc,
                                    double* __restrict__ vel_tmp) {
  double s_mp = 0.0, s_n = 0.0, s_p = 0.0, s_cnt = 0.0, s_v = 0.0, s_vcnt = 0.0;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_sel;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t f = sel ? sel[i] : i;
    const float* P = pred + f * J * 3;
    const float* G = gt + f * J * 3;
    // ---- mpjpe / n_mpjpe (fp32 like the reference's torch ops, sums in fp64)
    float npred = 0.f, ntar = 0.f, e1 = 0.f;
    for (int j = 0; j < J; ++j) {
      const float px = P[3 * j], py = P[3 * j + 1], pz = P[3 * j + 2];
      const float gx = G[3 * j], gy = G[3 * j + 1], gz = G[3 * j + 2];
      npred += px * px + py * py + pz * pz;
      ntar += gx * px + gy * py + gz * pz;
      const float dx = px - gx, dy = py - gy, dz = pz - gz;
      e1 += sqrtf(dx * dx + dy * dy + dz * dz);
    }
    const float scale = (ntar / J) / (npred / J);
    float e3 = 0.f;
    for (int j = 0; j < J; ++j) {
      const float dx = scale * P[3 * j] - G[3 * j], dy = scale * P[3 * j + 1] - G[3 * j + 1], dz = scale * P[3 * j + 2] - G[3 * j + 2];
      e3 += sqrtf(dx * dx + dy * dy + dz * dz);
    }
    // ---- p_mpjpe: X = target, Y = predicted (LOSS:50-79), fp64
    double muX[3] = {0, 0, 0}, muY[3] = {0, 0, 0};
    for (int j = 0; j < J; ++j)
      for (int c = 0; c < 3; ++c) { muX[c] += G[3 * j + c]; muY[c] += P[3 * j + c]; }
    for (int c = 0; c < 3; ++c) { muX[c] /= J; muY[c] /= J; }
    double nX = 0.0, nY = 0.0, H[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
    for (int j = 0; j < J; ++j) {
      double x[3], y[3];
      for (int c = 0; c < 3; ++c) { x[c] = G[3 * j + c] - muX[c]; y[c] = P[3 * j + c] - muY[c]; nX += x[c] * x[c]; nY += y[c] * y[c]; }
      for (int a = 0; a < 3; ++a)
        for (int b = 0; b < 3; ++b) H[a][b] += x[a] * y[b];          // X0^T Y0 (normalised below)
    }
    nX = sqrt(nX); nY = sqrt(nY);
    const double hn = 1.0 / (nX * nY);
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < 3; ++b) H[a][b] *= hn;
    // H = U S V^T  ->  H^T H = V S^2 V^T
    double A[3][3], V[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < 3; ++b) A[a][b] = H[0][a] * H[0][b] + H[1][a] * H[1][b] + H[2][a] * H[2][b];
    for (int sweep = 0; sweep < 12; ++sweep) {
      jacobi_rotate(A, V, 0, 1);
      jacobi_rotate(A, V, 0, 2);
      jacobi_rotate(A, V, 1, 2);
    }
    double lam[3] = {A[0][0], A[1][1], A[2][2]};
    int ord[3] = {0, 1, 2};                                           // descending singular values, as LAPACK returns them
    if (lam[ord[0]] < lam[ord[1]]) { int t = ord[0]; ord[0] = ord[1]; ord[1] = t; }
    if (lam[ord[1]] < lam[ord[2]]) { int t = ord[1]; ord[1] = ord[2]; ord[2] = t; }
    if (lam[ord[0]] < lam[ord[1]]) { int t = ord[0]; ord[0] = ord[1]; ord[1] = t; }
    double S[3], Vs[3][3], U[3][3];
    for (int k = 0; k < 3; ++k) {
      S[k] = sqrt(fmax(lam[ord[k]], 0.0));
      for (int a = 0; a < 3; ++a) Vs[a][k] = V[a][ord[k]];
    }
    for (int k = 0; k < 2; ++k) {                                     // U_k = H V_k / s_k
      double u[3], nu = 0.0;
      for (int a = 0; a < 3; ++a) { u[a] = H[a][0] * Vs[0][k] + H[a][1] * Vs[1][k] + H[a][2] * Vs[2][k]; nu += u[a] * u[a]; }
      nu = nu > 0.0 ? 1.0 / sqrt(nu) : 0.0;
      for (int a = 0; a < 3; ++a) U[a][k] = u[a] * nu;
    }
    {
      // third left vector: H V_3 / s_3 when s_3 is well above round-off, else the orthonormal completion (its sign
      // is fixed by the reflection test below either way)
      double u[3], nu = 0.0;
      for (int a = 0; a < 3; ++a) { u[a] = H[a][0] * Vs[0][2] + H[a][1] * Vs[1][2] + H[a][2] * Vs[2][2]; nu += u[a] * u[a]; }
      const double cx = U[1][0] * U[2][1] - U[2][0] * U[1][1], cy = U[2][0] * U[0][1] - U[0][0] * U[2][1],
                   cz = U[0][0] * U[1][1] - U[1][0] * U[0][1];
      if (S[2] > 1e-9 * S[0] && nu > 0.0) {
        nu = 1.0 / sqrt(nu);
        for (int a = 0; a < 3; ++a) U[a][2] = u[a] * nu;
      } else {
        U[0][2] = cx; U[1][2] = cy; U[2][2] = cz;
      }
    }
    // R = V U^T; reflection fix on the last column of V / last singular value (LOSS:66-70)
    auto det3 = [](const double (&m)[3][3]) {
      return m[0][0] * (m[1][1] * m[2][2] - m[1][2] * m[2][1]) - m[0][1] * (m[1][0] * m[2][2] - m[1][2] * m[2][0]) +
             m[0][2] * (m[1][0] * m[2][1] - m[1][1] * m[2][0]);
    };
    double R[3][3];
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < 3; ++b) R[a][b] = Vs[a][0] * U[b][0] + Vs[a][1] * U[b][1] + Vs[a][2] * U[b][2];
    const double dR = det3(R);
    const double sg = dR > 0.0 ? 1.0 : (dR < 0.0 ? -1.0 : 0.0);
    for (int a = 0; a < 3; ++a) Vs[a][2] *= sg;
    S[2] *= sg;
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < 3; ++b) R[a][b] = Vs[a][0] * U[b][0] + Vs[a][1] * U[b][1] + Vs[a][2] * U[b][2];
    const double tr = S[0] + S[1] + S[2];
    const double sc = tr * nX / nY;
    double t[3];
    for (int b = 0; b < 3; ++b) t[b] = muX[b] - sc * (muY[0] * R[0][b] + muY[1] * R[1][b] + muY[2] * R[2][b]);
    double e2 = 0.0;
    for (int j = 0; j < J; ++j) {
      double d2 = 0.0;
      for (int b = 0; b < 3; ++b) {
        const double al = sc * (P[3 * j] * R[0][b] + P[3 * j + 1] * R[1][b] + P[3 * j + 2] * R[2][b]) + t[b];
        const double d = al - G[3 * j + b];
        d2 += d * d;
      }
      e2 += sqrt(d2);
    }
    s_mp += e1; s_n += e3; s_p += e2; s_cnt += J;
    // ---- velocity error between this and the next selected frame (np.diff over the flattened batch, LOSS:139-142)
    if (i + 1 < n_sel) {
      const int64_t f2 = sel ? sel[i + 1] : i + 1;
      const float* P2 = pred + f2 * J * 3;
      const float* G2 = gt + f2 * J * 3;
      for (int j = 0; j < J; ++j) {
        const float dx = (P2[3 * j] - P[3 * j]) - (G2[3 * j] - G[3 * j]);
        const float dy = (P2[3 * j + 1] - P[3 * j + 1]) - (G2[3 * j + 1] - G[3 * j + 1]);
        const float dz = (P2[3 * j + 2] - P[3 * j + 2]) - (G2[3 * j + 2] - G[3 * j + 2]);
        s_v += sqrtf(dx * dx + dy * dy + dz * dz);
      }
      s_vcnt += J;
    }
  }
  double vals[6] = {s_mp, s_n, s_p, s_cnt, s_v, s_vcnt};
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    double v = vals[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    // the velocity pair is per CALL: finalised with the reference's weighting by vel_finalize_kernel
    if ((threadIdx.x & 31) == 0 && v != 0.0) atomicAdd(k < 4 ? acc + k : vel_tmp + (k - 4), v);
  }
}

// evaluate() weights every batch's mean velocity error by its frame count (RUN:610-614:
// `epoch_loss_3d_vel += N_b * mean_velocity_error(batch)`, divided by sum N_b at the end), and the mean inside a batch
// runs over its (N_b - 1) * J frame differences (LOSS:139-142): acc[4] += N_b * tmp[0] / tmp[1], acc[5] += N_b.
__global__ void vel_finalize_kernel(double* __restrict__ acc, double* __restrict__ vel_tmp, double n_frames) {
  if (vel_tmp[1] > 0.0) acc[4] += n_frames * (vel_tmp[0] / vel_tmp[1]);
  acc[5] += n_frames;
  vel_tmp[0] = 0.0;
  vel_tmp[1] = 0.0;
}

// MPI-INF-3DHP PCK / AUC (d3d_pck_accumulate): a grouped, per-joint histogram of joint errors.  The protocol (thresholds,
// evaluated joints, units) is the caller's; the kernel only counts.  One warp per listed frame, lane j = joint j.
// The error is d = sqrt((dx*dx + dy*dy) + dz*dz), dx = pred - gt, rounded after every operation (no FMA contraction) so
// that a float32 restatement on the host reproduces it bit for bit.  Its bin b is the number of thresholds d is NOT
// below (strict <): the joint counts under thresholds b..n-1.  NaN and +inf land in bin n and count under none.
// kSmem: the block builds [n_groups][J][n] per-bin counts in shared memory and adds their prefix sums to `counts` at
// exit, one atomic per non-zero (group, joint, threshold).  Otherwise every joint adds 1 to counts[g][j][b..n-1] directly.
// The error and frame sums of a lane stay in registers while consecutive frames of the warp share a group.
template <bool kSmem>
__global__ void __launch_bounds__(512) pck_hist_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                                       const int64_t* __restrict__ sel, const int32_t* __restrict__ group,
                                                       int64_t n_sel, int J, const __grid_constant__ PckThresholds thr,
                                                       int n_groups, unsigned long long* __restrict__ counts,
                                                       double* __restrict__ err_sum,
                                                       unsigned long long* __restrict__ frames) {
  extern __shared__ unsigned int bins[];               // kSmem: [n_groups][J][n]
  __shared__ float s_thr[kPckMaxThresholds];           // padded with +inf for the fixed-depth search
  const int n = thr.n;
  const int rows = n_groups * J;
  if (threadIdx.x < kPckMaxThresholds) s_thr[threadIdx.x] = threadIdx.x < n ? thr.t[threadIdx.x] : __int_as_float(0x7f800000);
  if (kSmem)
    for (int i = threadIdx.x; i < rows * n; i += blockDim.x) bins[i] = 0u;
  __syncthreads();

  const int lane = threadIdx.x & 31;
  const int64_t n_warps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  int cur = -1;                                        // group whose sums this lane holds
  double esum = 0.0;
  unsigned long long nf = 0;
  auto flush = [&]() {
    if (cur < 0) return;
    if (lane < J) atomicAdd(err_sum + static_cast<int64_t>(cur) * J + lane, esum);
    if (lane == 0) atomicAdd(frames + cur, nf);
  };
  for (int64_t i = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; i < n_sel; i += n_warps) {
    const int64_t f = sel ? sel[i] : i;
    const int g = group ? group[f] : 0;
    if (g < 0 || g >= n_groups) continue;              // warp-uniform: the whole frame is skipped
    if (g != cur) {
      flush();
      cur = g;
      esum = 0.0;
      nf = 0;
    }
    ++nf;
    if (lane < J) {
      const float* P = pred + (f * J + lane) * 3;
      const float* G = gt + (f * J + lane) * 3;
      const float dx = __fsub_rn(P[0], G[0]), dy = __fsub_rn(P[1], G[1]), dz = __fsub_rn(P[2], G[2]);
      const float d = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
      esum += static_cast<double>(d);
      // b = #{k : !(d < s_thr[k])}: the predicate is true on a prefix of the 64 padded thresholds
      int b = 0;
#pragma unroll
      for (int step = 32; step > 0; step >>= 1)
        if (!(d < s_thr[b + step - 1])) b += step;
      if (!(d < s_thr[b])) ++b;                         // b <= 63 here
      if (b < n) {
        const int64_t row = static_cast<int64_t>(g) * J + lane;
        if (kSmem) {
          atomicAdd(bins + row * n + b, 1u);
        } else {
          for (int k = b; k < n; ++k) atomicAdd(counts + row * n + k, 1ull);
        }
      }
    }
  }
  flush();
  if (kSmem) {
    __syncthreads();
    for (int r = threadIdx.x; r < rows; r += blockDim.x) {
      unsigned long long run = 0;
      for (int k = 0; k < n; ++k) {
        run += bins[r * n + k];
        if (run) atomicAdd(counts + static_cast<int64_t>(r) * n + k, run);
      }
    }
  }
}

}  // namespace

cudaError_t launch_pose_metrics(const float* pred, const float* gt, const int64_t* sel, int64_t n_sel, int J, double* acc,
                                double* vel_tmp, cudaStream_t st) {
  if (n_sel <= 0) return cudaSuccess;
  if (J < 1 || J > kMaxJ) return cudaErrorInvalidValue;
  int64_t g = (n_sel + 127) / 128;
  if (g > 148 * 16) g = 148 * 16;
  pose_metrics_kernel<<<static_cast<unsigned>(g), 128, 0, st>>>(pred, gt, sel, n_sel, J, acc, vel_tmp);
  vel_finalize_kernel<<<1, 1, 0, st>>>(acc, vel_tmp, static_cast<double>(n_sel));
  return cudaGetLastError();
}

cudaError_t launch_pck_hist(const float* pred, const float* gt, const int64_t* sel, const int32_t* group, int64_t n_sel,
                            int J, const PckThresholds& thr, int n_groups, int64_t* counts, double* err_sum,
                            int64_t* frames, int num_sms, cudaStream_t st) {
  if (n_sel <= 0) return cudaSuccess;
  if (J < 1 || J > kMaxJ || thr.n < 1 || thr.n > kPckMaxThresholds || n_groups < 1 || n_groups > kPckMaxGroups)
    return cudaErrorInvalidValue;
  constexpr int kThreads = 512;
  // two blocks per SM: the shared-memory path pays one flush of its whole histogram per block
  int64_t g = (n_sel + kThreads / 32 - 1) / (kThreads / 32);
  if (g > 2 * num_sms) g = 2 * num_sms;
  const int64_t bin_bytes = static_cast<int64_t>(n_groups) * J * thr.n * sizeof(unsigned int);
  auto* c = reinterpret_cast<unsigned long long*>(counts);
  auto* fr = reinterpret_cast<unsigned long long*>(frames);
  if (bin_bytes <= kPckSmemBinBytes)
    pck_hist_kernel<true><<<static_cast<unsigned>(g), kThreads, static_cast<size_t>(bin_bytes), st>>>(
        pred, gt, sel, group, n_sel, J, thr, n_groups, c, err_sum, fr);
  else
    pck_hist_kernel<false><<<static_cast<unsigned>(g), kThreads, 0, st>>>(pred, gt, sel, group, n_sel, J, thr, n_groups,
                                                                          c, err_sum, fr);
  return cudaGetLastError();
}

}  // namespace d3d
