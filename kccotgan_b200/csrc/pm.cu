// Martingale penalty p_M (gan_utils.py:179-201) and its gradient.
//   N = M[:,1:] - M[:,:-1];  sigma_j = population std of M[:,:,j];  A_tj = (1/m) sum_i N_itj / (sigma_j + 1e-6)
//   p_M = lam * s * sum_tj |A_tj|
#include "common.cuh"

namespace kccot {
namespace {
constexpr int PT = 256;

// one CTA; thread e walks column e of the [B, T*J] matrix (coalesced across e).  The single and the batched
// kernels inline this one body, so each problem of a batched call gets the single call's instructions and bits.
__device__ __forceinline__ void pm_fwd_cta(const float* __restrict__ M, int B, int T, int J, float w,
                                           float* __restrict__ pm, float* __restrict__ stats) {
  extern __shared__ float sh[];          // S[TJ] | V[TJ] | mean[J] | den[J] | red[32]
  const int TJ = T * J;
  float* S = sh;
  float* V = sh + TJ;
  float* mean = V + TJ;
  float* den = mean + J;
  float* red = den + J;
  for (int e = threadIdx.x; e < TJ; e += PT) {
    float a = 0.f;
    for (int i = 0; i < B; ++i) a += M[(long long)i * TJ + e];
    S[e] = a;
  }
  __syncthreads();
  for (int j = threadIdx.x; j < J; j += PT) {
    float a = 0.f;
    for (int t = 0; t < T; ++t) a += S[t * J + j];
    mean[j] = a / ((float)B * (float)T);
  }
  __syncthreads();
  for (int e = threadIdx.x; e < TJ; e += PT) {
    const float mu = mean[e % J];
    float a = 0.f, d = 0.f;
    const bool has_next = e < TJ - J;
    for (int i = 0; i < B; ++i) {
      const float x = M[(long long)i * TJ + e];
      a = fmaf(x - mu, x - mu, a);
      if (has_next) d += M[(long long)i * TJ + e + J] - x;
    }
    V[e] = a;
    S[e] = d;                             // now: sum_i N[i, t, j]
  }
  __syncthreads();
  for (int j = threadIdx.x; j < J; j += PT) {
    float a = 0.f;
    for (int t = 0; t < T; ++t) a += V[t * J + j];
    const float sd = sqrtf(a / ((float)B * (float)T));
    den[j] = sd + 1e-6f;
    stats[j] = mean[j];
    stats[J + j] = sd;
  }
  __syncthreads();
  float acc = 0.f;
  for (int e = threadIdx.x; e < TJ - J; e += PT) {
    const float A = S[e] / (float)B / den[e % J];
    stats[2 * J + e] = A;
    acc += fabsf(A);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f;
    for (int q = 0; q < PT / 32; ++q) a += red[q];
    *pm = w * a;
  }
}

__global__ void __launch_bounds__(PT) pm_fwd_kernel(const float* __restrict__ M, int B, int T, int J, float w,
                                                    float* __restrict__ pm, float* __restrict__ stats) {
  pm_fwd_cta(M, B, T, J, w, pm, stats);
}

// problem blockIdx.x of M [nprob, B, T, J]: pm[p] and stats row p [2J + (T-1)J]
__global__ void __launch_bounds__(PT) pm_batched_fwd_kernel(const float* __restrict__ M, int B, int T, int J, float w,
                                                            float* __restrict__ pm, float* __restrict__ stats) {
  const int p = blockIdx.x;
  pm_fwd_cta(M + (long long)p * B * T * J, B, T, J, w, pm + p, stats + (long long)p * (2 * J + (T - 1) * J));
}

// element idx < B*T*J of one problem
__device__ __forceinline__ void pm_bwd_elem(const float* __restrict__ M, int B, int T, int J, float w,
                                            const float* __restrict__ stats, const float* __restrict__ gpm,
                                            float* __restrict__ gM, long long idx) {
  const int j = (int)(idx % J), t = (int)((idx / J) % T);
  const float mu = stats[j], sd = stats[J + j], den = sd + 1e-6f;
  const float* A = stats + 2 * J;
  const float g = *gpm * w;
  auto sgn = [](float a) { return (a > 0.f) ? 1.f : ((a < 0.f) ? -1.f : 0.f); };
  float v = 0.f;
  if (t >= 1) v += sgn(A[(t - 1) * J + j]);
  if (t <= T - 2) v -= sgn(A[t * J + j]);
  v = v / ((float)B * den);
  float absA = 0.f;
  for (int tt = 0; tt < T - 1; ++tt) absA += fabsf(A[tt * J + j]);
  const float gsig = -absA / den;
  if (sd > 0.f) v += gsig * (M[idx] - mu) / ((float)B * (float)T * sd);
  gM[idx] = g * v;
}

__global__ void __launch_bounds__(PT) pm_bwd_kernel(const float* __restrict__ M, int B, int T, int J, float w,
                                                    const float* __restrict__ stats, const float* __restrict__ gpm,
                                                    float* __restrict__ gM) {
  const long long n = (long long)B * T * J;
  const long long idx = (long long)blockIdx.x * PT + threadIdx.x;
  if (idx >= n) return;
  pm_bwd_elem(M, B, T, J, w, stats, gpm, gM, idx);
}

// grid (ceil(B*T*J / PT), nprob): problem blockIdx.y reads its own stats row and gpm[p]
__global__ void __launch_bounds__(PT) pm_batched_bwd_kernel(const float* __restrict__ M, int B, int T, int J, float w,
                                                            const float* __restrict__ stats,
                                                            const float* __restrict__ gpm, float* __restrict__ gM) {
  const long long n = (long long)B * T * J;
  const long long idx = (long long)blockIdx.x * PT + threadIdx.x;
  if (idx >= n) return;
  const int p = blockIdx.y;
  pm_bwd_elem(M + p * n, B, T, J, w, stats + (long long)p * (2 * J + (T - 1) * J), gpm + p, gM + p * n, idx);
}
}  // namespace
}  // namespace kccot

using namespace kccot;

extern "C" {
int kccot_pm_fwd(const float* M, int B, int T, int J, float reg_lam, float s, float* pm, float* stats, void* stream) {
  KCCOT_CHECK_ARG(M && pm && stats, "null pointer");
  KCCOT_CHECK_ARG(B >= 1 && T >= 2 && J >= 1, "bad sizes B=%d T=%d J=%d", B, T, J);
  const size_t smem = (size_t)(2 * T * J + 2 * J + 32) * sizeof(float);
  KCCOT_CHECK_ARG(smem <= 48 * 1024, "T*J too large for the p_M kernel (%d)", T * J);
  pm_fwd_kernel<<<1, PT, smem, (cudaStream_t)stream>>>(M, B, T, J, reg_lam * s, pm, stats);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}
int kccot_pm_bwd(const float* M, int B, int T, int J, float reg_lam, float s, const float* stats, const float* gpm,
                 float* gM, void* stream) {
  KCCOT_CHECK_ARG(M && stats && gpm && gM, "null pointer");
  KCCOT_CHECK_ARG(B >= 1 && T >= 2 && J >= 1, "bad sizes");
  const long long n = (long long)B * T * J;
  pm_bwd_kernel<<<(unsigned)((n + PT - 1) / PT), PT, 0, (cudaStream_t)stream>>>(M, B, T, J, reg_lam * s, stats, gpm, gM);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}
int kccot_pm_batched_fwd(const float* M, int nprob, int B, int T, int J, float reg_lam, float s, float* pm,
                         float* stats, void* stream) {
  KCCOT_CHECK_ARG(M && pm && stats, "null pointer");
  KCCOT_CHECK_ARG(nprob >= 1 && nprob <= 65535, "nprob=%d outside 1..65535", nprob);
  KCCOT_CHECK_ARG(B >= 1 && T >= 2 && J >= 1, "bad sizes B=%d T=%d J=%d", B, T, J);
  const size_t smem = (size_t)(2 * T * J + 2 * J + 32) * sizeof(float);
  KCCOT_CHECK_ARG(smem <= 48 * 1024, "T*J too large for the p_M kernel (%d)", T * J);
  pm_batched_fwd_kernel<<<nprob, PT, smem, (cudaStream_t)stream>>>(M, B, T, J, reg_lam * s, pm, stats);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}
int kccot_pm_batched_bwd(const float* M, int nprob, int B, int T, int J, float reg_lam, float s, const float* stats,
                         const float* gpm, float* gM, void* stream) {
  KCCOT_CHECK_ARG(M && stats && gpm && gM, "null pointer");
  KCCOT_CHECK_ARG(nprob >= 1 && nprob <= 65535, "nprob=%d outside 1..65535", nprob);
  KCCOT_CHECK_ARG(B >= 1 && T >= 2 && J >= 1, "bad sizes B=%d T=%d J=%d", B, T, J);
  const long long n = (long long)B * T * J;
  const dim3 grid((unsigned)((n + PT - 1) / PT), (unsigned)nprob);
  pm_batched_bwd_kernel<<<grid, PT, 0, (cudaStream_t)stream>>>(M, B, T, J, reg_lam * s, stats, gpm, gM);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}
}
