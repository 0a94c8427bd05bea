// Pre- and post-passes of the large-batch cost path (B > 64) around gemm_f16x3.cu.  All HBM-bound
// streaming kernels; none is on the critical path at config 5 (the GEMMs take > 90 % of the time).
//
//   forward  (gan_utils.py:14-17 in GEMM form, :34-38 for the martingale term):
//     colsum_part / colmean : column means c_k of the stacked rows Z = [x; y] and max|z| (-> power-of-two scale)
//     split                 : z~ = (z - c) * 2^e  ->  fp16 hi = rn(z~), lo = rn(z~ - hi), row-major [R][Kp]
//     rownorm               : n_i = sum_k (hi + lo)^2 (the represented values), fp64 block reduction
//     [gemm_f16x3]          : P_ij = sum_k z~_i z~_j  (raw dot products, split-K partials)
//     finalize              : C_ij = s (n_i + n_j - 2 P_ij) / 4^e + s sum_q h_i,q dM_j,q ; symmetric blocks are
//                             mirrored from the computed upper-triangle tiles, self-cost diagonals are exactly 0
//   backward (adjoint of the same lines; W' = W - diag(rowsum W) as in grad_tcgen05.cu):
//     w_tiles / w_rowsum / w_convert : W' from the cost adjoints, scaled by a power of two, fp16 hi/lo [rows][Rp]
//     split (transposed)    : ZT [Kp][Rp] fp16 hi/lo, so that the adjoint is the same K-major x K-major GEMM
//     [gemm_f16x3]          : g = -2 s / (2^e 2^f) * W'_scaled . z~_scaled   (rows of W' sum to zero, so the
//                             centre c drops out exactly as in the reference's (x_i - y_j) form)
#include <cuda_fp16.h>

#include "cost.cuh"
#include "large.cuh"

namespace kccot {

namespace {
__device__ __forceinline__ float pow2f(int e) {          // 2^e for e in [-126, 127]
  e = max(-126, min(127, e));
  return __int_as_float((e + 127) << 23);
}
__device__ __forceinline__ int floor_log2_bits(unsigned bits) {   // of a positive finite float given by its bits
  return max(-100, min(100, (int)((bits >> 23) & 0xffu) - 127));
}

// ---- column sums -------------------------------------------------------------------------------
// grid (ceil(K / 128), nseg): thread = one column, CTA = 128 columns x one row segment.  part[seg][k].
__global__ void __launch_bounds__(128) colsum_part_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                                          int Bx, int By, long long K, int rows_per_seg,
                                                          float* __restrict__ part, unsigned* __restrict__ absmax) {
  const long long k = (long long)blockIdx.x * 128 + threadIdx.x;
  const int R = Bx + By;
  const int r0 = blockIdx.y * rows_per_seg, r1 = min(R, r0 + rows_per_seg);
  float acc = 0.f, mx = 0.f;
  if (k < K) {
    int r = r0;
    for (; r + 4 <= r1; r += 4) {
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int rr = r + u;
        v[u] = (rr < Bx) ? x[(long long)rr * K + k] : y[(long long)(rr - Bx) * K + k];
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) { acc += v[u]; mx = fmaxf(mx, fabsf(v[u])); }
    }
    for (; r < r1; ++r) {
      const float v = (r < Bx) ? x[(long long)r * K + k] : y[(long long)(r - Bx) * K + k];
      acc += v;
      mx = fmaxf(mx, fabsf(v));
    }
    part[(long long)blockIdx.y * K + k] = acc;
  }
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0 && mx > 0.f && mx < 3.0e38f) atomicMax(absmax, __float_as_uint(mx));
}

// mean[k] = sum_seg part / R ; block 0 also derives the power-of-two scale of the split from max|z|
__global__ void __launch_bounds__(256) colmean_kernel(const float* __restrict__ part, int nseg, long long K, int R,
                                                      float* __restrict__ mean, float* __restrict__ scal) {
  const long long k = (long long)blockIdx.x * 256 + threadIdx.x;
  if (k < K) {
    float acc = 0.f;
    for (int s = 0; s < nseg; ++s) acc += part[(long long)s * K + k];
    mean[k] = acc / (float)R;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const unsigned bits = reinterpret_cast<const unsigned*>(scal)[kScalAbsmax];
    int e = 0;
    if (bits != 0) e = 12 - floor_log2_bits(bits);          // |z - c| <= 2 max|z| < 2^(ex + 2)  ->  < 2^14 after scaling
    scal[kScalZscale] = pow2f(e);
    scal[kScalZinv] = pow2f(-e);
  }
}

// ---- centre, scale, split -----------------------------------------------------------------------
// grid (ceil(K / 64), ceil(R / 64)), 256 threads, tile 64 rows x 64 columns.
__global__ void __launch_bounds__(256) split_kernel(const float* __restrict__ x, const float* __restrict__ y, int Bx,
                                                    int By, long long K, long long Kp, int Rp,
                                                    const float* __restrict__ mean, const float* __restrict__ scal,
                                                    __half* __restrict__ Zh1, __half* __restrict__ Zh2,
                                                    __half* __restrict__ ZT1, __half* __restrict__ ZT2) {
  __shared__ __half t1[64][72], t2[64][72];                 // [column][row] for the transposed copy
  const int R = Bx + By;
  const long long c0 = (long long)blockIdx.x * 64;
  const int r0 = blockIdx.y * 64;
  const int t = threadIdx.x;
  const int cg = (t & 15) * 4;
  const float zs = scal[kScalZscale];
  float m[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) m[e] = (c0 + cg + e < K) ? mean[c0 + cg + e] : 0.f;
  const bool vec = ((K & 3) == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(y) & 15) == 0);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int rl = (t >> 4) + 16 * i;
    const int r = r0 + rl;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (r < R) {
      const float* src = (r < Bx) ? x + (long long)r * K : y + (long long)(r - Bx) * K;
      if (vec && c0 + cg + 3 < K) {
        const float4 q = *reinterpret_cast<const float4*>(src + c0 + cg);
        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (c0 + cg + e < K) v[e] = src[c0 + cg + e];
      }
    }
    __half h1[4], h2[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const bool in = (r < R) && (c0 + cg + e < K);
      const float z = in ? (v[e] - m[e]) * zs : 0.f;
      h1[e] = __float2half_rn(z);
      h2[e] = __float2half_rn(z - __half2float(h1[e]));
    }
    if (Zh1 != nullptr && r < R && c0 + cg < Kp) {          // Kp is a multiple of 64: the 4-group is inside the pitch
      *reinterpret_cast<uint2*>(Zh1 + (long long)r * Kp + c0 + cg) = *reinterpret_cast<const uint2*>(h1);
      *reinterpret_cast<uint2*>(Zh2 + (long long)r * Kp + c0 + cg) = *reinterpret_cast<const uint2*>(h2);
    }
    if (ZT1 != nullptr) {
#pragma unroll
      for (int e = 0; e < 4; ++e) { t1[cg + e][rl] = h1[e]; t2[cg + e][rl] = h2[e]; }
    }
  }
  if (ZT1 == nullptr) return;
  __syncthreads();
  // transposed rows: 4 threads per video column, 16 stacked rows (32 bytes) each
  const int c = t >> 2, seg = (t & 3) * 16;
  if (c0 + c < Kp && r0 + seg < Rp) {                        // Rp is a multiple of 64
    const uint4* s1 = reinterpret_cast<const uint4*>(&t1[c][seg]);
    const uint4* s2 = reinterpret_cast<const uint4*>(&t2[c][seg]);
    uint4* d1 = reinterpret_cast<uint4*>(ZT1 + (c0 + c) * (long long)Rp + r0 + seg);
    uint4* d2 = reinterpret_cast<uint4*>(ZT2 + (c0 + c) * (long long)Rp + r0 + seg);
    d1[0] = s1[0]; d1[1] = s1[1];
    d2[0] = s2[0]; d2[1] = s2[1];
  }
}

// ---- bf16 videos ---------------------------------------------------------------------------------
// colsum_part_kernel and split_kernel for bf16 videos (raw bits).  A bf16 value widens exactly, so after the load
// each runs the fp32 kernel's instruction sequence and summation order: the column sums, the scale and the fp16 split
// equal the fp32 kernels' on the widened videos.  Separate kernels, so that the fp32 ones keep their code.
__device__ __forceinline__ float ld1(const uint16_t* __restrict__ p, long long i) {
  return __uint_as_float((unsigned)p[i] << 16);
}

__global__ void __launch_bounds__(128) colsum_part_bf16_kernel(const uint16_t* __restrict__ x,
                                                               const uint16_t* __restrict__ y, int Bx, int By,
                                                               long long K, int rows_per_seg, float* __restrict__ part,
                                                               unsigned* __restrict__ absmax) {
  const long long k = (long long)blockIdx.x * 128 + threadIdx.x;
  const int R = Bx + By;
  const int r0 = blockIdx.y * rows_per_seg, r1 = min(R, r0 + rows_per_seg);
  float acc = 0.f, mx = 0.f;
  if (k < K) {
    int r = r0;
    for (; r + 4 <= r1; r += 4) {
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int rr = r + u;
        v[u] = (rr < Bx) ? ld1(x, (long long)rr * K + k) : ld1(y, (long long)(rr - Bx) * K + k);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) { acc += v[u]; mx = fmaxf(mx, fabsf(v[u])); }
    }
    for (; r < r1; ++r) {
      const float v = (r < Bx) ? ld1(x, (long long)r * K + k) : ld1(y, (long long)(r - Bx) * K + k);
      acc += v;
      mx = fmaxf(mx, fabsf(v));
    }
    part[(long long)blockIdx.y * K + k] = acc;
  }
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0 && mx > 0.f && mx < 3.0e38f) atomicMax(absmax, __float_as_uint(mx));
}

__global__ void __launch_bounds__(256) split_bf16_kernel(const uint16_t* __restrict__ x, const uint16_t* __restrict__ y,
                                                         int Bx, int By, long long K, long long Kp, int Rp,
                                                         const float* __restrict__ mean, const float* __restrict__ scal,
                                                         __half* __restrict__ Zh1, __half* __restrict__ Zh2,
                                                         __half* __restrict__ ZT1, __half* __restrict__ ZT2) {
  __shared__ __half t1[64][72], t2[64][72];                 // [column][row] for the transposed copy
  const int R = Bx + By;
  const long long c0 = (long long)blockIdx.x * 64;
  const int r0 = blockIdx.y * 64;
  const int t = threadIdx.x;
  const int cg = (t & 15) * 4;
  const float zs = scal[kScalZscale];
  float m[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) m[e] = (c0 + cg + e < K) ? mean[c0 + cg + e] : 0.f;
  const bool vec = ((K & 3) == 0) && ((reinterpret_cast<uintptr_t>(x) & 7) == 0) &&
                   ((reinterpret_cast<uintptr_t>(y) & 7) == 0);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int rl = (t >> 4) + 16 * i;
    const int r = r0 + rl;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (r < R) {
      const uint16_t* src = (r < Bx) ? x + (long long)r * K : y + (long long)(r - Bx) * K;
      if (vec && c0 + cg + 3 < K) {
        const float4 q = widen_bf16x4(*reinterpret_cast<const uint2*>(src + c0 + cg));
        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (c0 + cg + e < K) v[e] = ld1(src, c0 + cg + e);
      }
    }
    __half h1[4], h2[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const bool in = (r < R) && (c0 + cg + e < K);
      const float z = in ? (v[e] - m[e]) * zs : 0.f;
      h1[e] = __float2half_rn(z);
      h2[e] = __float2half_rn(z - __half2float(h1[e]));
    }
    if (Zh1 != nullptr && r < R && c0 + cg < Kp) {          // Kp is a multiple of 64: the 4-group is inside the pitch
      *reinterpret_cast<uint2*>(Zh1 + (long long)r * Kp + c0 + cg) = *reinterpret_cast<const uint2*>(h1);
      *reinterpret_cast<uint2*>(Zh2 + (long long)r * Kp + c0 + cg) = *reinterpret_cast<const uint2*>(h2);
    }
    if (ZT1 != nullptr) {
#pragma unroll
      for (int e = 0; e < 4; ++e) { t1[cg + e][rl] = h1[e]; t2[cg + e][rl] = h2[e]; }
    }
  }
  if (ZT1 == nullptr) return;
  __syncthreads();
  // transposed rows: 4 threads per video column, 16 stacked rows (32 bytes) each
  const int c = t >> 2, seg = (t & 3) * 16;
  if (c0 + c < Kp && r0 + seg < Rp) {                        // Rp is a multiple of 64
    const uint4* s1 = reinterpret_cast<const uint4*>(&t1[c][seg]);
    const uint4* s2 = reinterpret_cast<const uint4*>(&t2[c][seg]);
    uint4* d1 = reinterpret_cast<uint4*>(ZT1 + (c0 + c) * (long long)Rp + r0 + seg);
    uint4* d2 = reinterpret_cast<uint4*>(ZT2 + (c0 + c) * (long long)Rp + r0 + seg);
    d1[0] = s1[0]; d1[1] = s1[1];
    d2[0] = s2[0]; d2[1] = s2[1];
  }
}

// ---- row norms of the represented values ----------------------------------------------------------
__global__ void __launch_bounds__(256) rownorm_kernel(const __half* __restrict__ Zh1, const __half* __restrict__ Zh2,
                                                      long long K, long long Kp, float* __restrict__ norms) {
  const int r = blockIdx.x;
  const uint4* a = reinterpret_cast<const uint4*>(Zh1 + (long long)r * Kp);
  const uint4* b = reinterpret_cast<const uint4*>(Zh2 + (long long)r * Kp);
  const long long n8 = K >> 3;
  double acc = 0.0;
  for (long long i = threadIdx.x; i < n8; i += 256) {
    const uint4 qa = a[i], qb = b[i];
    const __half2* ha = reinterpret_cast<const __half2*>(&qa);
    const __half2* hb = reinterpret_cast<const __half2*>(&qb);
    float p = 0.f;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 fa = __half22float2(ha[e]), fb = __half22float2(hb[e]);
      const float z0 = fa.x + fb.x, z1 = fa.y + fb.y;
      p = fmaf(z0, z0, fmaf(z1, z1, p));
    }
    acc += (double)p;
  }
  for (long long k = (n8 << 3) + threadIdx.x; k < K; k += 256) {
    const float z = __half2float(Zh1[(long long)r * Kp + k]) + __half2float(Zh2[(long long)r * Kp + k]);
    acc += (double)(z * z);
  }
  __shared__ double red[8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += red[w];
    norms[r] = (float)s;
  }
}

// ---- finalize ------------------------------------------------------------------------------------
constexpr int FQ = 32;     // martingale contraction chunk

__global__ void __launch_bounds__(256) large_finalize_kernel(LargeFin F, int T, int J, float s,
                                                             const float* __restrict__ scal) {
  // one buffer, two uses: the martingale operand tiles (2 x 64 x (FQ+1) floats), then the transposed source
  // tile of a mirrored block (64 x 65 doubles)
  __shared__ double sbuf[64 * 65];
  float (*hs)[FQ + 1] = reinterpret_cast<float (*)[FQ + 1]>(sbuf);
  float (*ms)[FQ + 1] = hs + 64;
  double (*pt)[65] = reinterpret_cast<double (*)[65]>(sbuf);
  const LargeFinBlock& b = F.b[blockIdx.z];
  const int i0 = blockIdx.y * 64, j0 = blockIdx.x * 64;
  if (i0 >= b.Bx || j0 >= b.By) return;
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const float zinv = scal[kScalZinv];
  float mart[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int c = 0; c < 4; ++c) mart[a][c] = 0.f;
  const int TJ = T * J, Q = (T - 1) * J;
  for (int pair = 0; pair < 2; ++pair) {
    const float* h = pair ? b.h2 : b.h1;
    const float* M = pair ? b.M2 : b.M1;
    if (h == nullptr) continue;
    for (int q0 = 0; q0 < Q; q0 += FQ) {
      __syncthreads();
      for (int e = t; e < 64 * FQ; e += 256) {
        const int rr = e / FQ, q = q0 + e % FQ;
        float hv = 0.f, mv = 0.f;
        if (q < Q) {
          if (i0 + rr < b.Bx) hv = h[(long long)(i0 + rr) * TJ + q];
          if (j0 + rr < b.By) {
            const float* mp = M + (long long)(j0 + rr) * TJ + q;
            mv = mp[J] - mp[0];
          }
        }
        hs[rr][e % FQ] = hv;
        ms[rr][e % FQ] = mv;
      }
      __syncthreads();
#pragma unroll 8
      for (int q = 0; q < FQ; ++q) {
        float hv[4], mv[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) { hv[a] = hs[ty * 4 + a][q]; mv[a] = ms[tx * 4 + a][q]; }
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int c = 0; c < 4; ++c) mart[a][c] = fmaf(hv[a], mv[c], mart[a][c]);
      }
    }
  }
  // Symmetric blocks hold only the 256 x 256 tiles on or above the diagonal (uniform over this 64 x 64 tile):
  // the rest is the mirror image, read along ITS rows (coalesced) and transposed through shared memory.
  const bool stored = !b.tri || ((j0 / G3_BN) >= (i0 / G3_BN));
  if (!stored) {
    __syncthreads();                                     // hs / ms are dead
    for (int e = t; e < 64 * 64; e += 256) {
      const int jj = e >> 6, ii = e & 63;                // source row j0 + jj, source column i0 + ii
      double d = 0.0;
      if (j0 + jj < b.By && i0 + ii < b.Bx) {
        const float* pp = b.P + (long long)(j0 + jj) * b.ld + i0 + ii;
        for (int ks = 0; ks < b.nks; ++ks) d += (double)pp[(long long)ks * b.ks_stride];
      }
      pt[jj][ii] = d;
    }
    __syncthreads();
  }
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int i = i0 + ty * 4 + a;
    if (i >= b.Bx) continue;
    const float ni = b.ni[i];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int j = j0 + tx * 4 + c;
      if (j >= b.By) continue;
      float out;
      if (b.zero_diag && i + b.diag_off == j) {
        out = s * mart[a][c];
      } else {
        double d = 0.0;
        if (stored) {
          const float* pp = b.P + (long long)i * b.ld + j;
          for (int ks = 0; ks < b.nks; ++ks) d += (double)pp[(long long)ks * b.ks_stride];
        } else {
          d = pt[tx * 4 + c][ty * 4 + a];
        }
        const double D = ((double)ni + (double)b.nj[j] - 2.0 * d) * (double)zinv * (double)zinv;
        out = s * (float)D + s * mart[a][c];
      }
      b.C[(long long)i * b.ldc + j] = out;
    }
  }
}

// ---- W' ------------------------------------------------------------------------------------------
// value of the symmetric weight matrix W at (r, c) without the diagonal, split into the term read along
// the row (direct) and the term read along the column (transposed)
struct WSrc {
  const float *Cxx, *Cxy, *Cyy;
  int Bx, By;
  // row-shard mode (XYcol != nullptr): only fake rows [row0, row0 + nloc) exist, as column panels / own rows
  const float *XYcol, *YYcol, *YYrow;
  int row0, nloc;
};
__device__ __forceinline__ float w_direct(const WSrc& S, int r, int c) {
  if (S.XYcol != nullptr) {
    if (c < S.Bx) return 0.f;
    return S.YYrow[(long long)(r - S.Bx - S.row0) * S.By + (c - S.Bx)];
  }
  if (r < S.Bx) {
    if (c < S.Bx) return S.Cxx ? S.Cxx[(long long)r * S.Bx + c] : 0.f;
    return S.Cxy[(long long)r * S.By + (c - S.Bx)];
  }
  if (c < S.Bx) return 0.f;
  return S.Cyy ? S.Cyy[(long long)(r - S.Bx) * S.By + (c - S.Bx)] : 0.f;
}
__device__ __forceinline__ float w_transposed(const WSrc& S, int r, int c) {
  if (S.XYcol != nullptr) {
    const int jl = r - S.Bx - S.row0;
    if (c < S.Bx) return S.XYcol[(long long)c * S.nloc + jl];
    return S.YYcol[(long long)(c - S.Bx) * S.nloc + jl];
  }
  if (r < S.Bx) {
    if (c < S.Bx) return S.Cxx ? S.Cxx[(long long)c * S.Bx + r] : 0.f;
    return 0.f;
  }
  if (c < S.Bx) return S.Cxy[(long long)c * S.By + (r - S.Bx)];
  return S.Cyy ? S.Cyy[(long long)(c - S.Bx) * S.By + (r - S.Bx)] : 0.f;
}

// grid (ceil(R / 32), ceil(nrows / 32)), block (32, 8)
__global__ void __launch_bounds__(256) w_tiles_kernel(WSrc S, int row_off, int nrows, int Rp, float* __restrict__ Wtmp,
                                                      float* __restrict__ rs_part, unsigned* __restrict__ wabs) {
  __shared__ float tt[32][33];
  const int R = S.Bx + S.By;
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int cb = blockIdx.x * 32, rb = blockIdx.y * 32;
  for (int cc = ty; cc < 32; cc += 8) {
    const int c = cb + cc, rl = rb + tx;
    tt[cc][tx] = (c < R && rl < nrows) ? w_transposed(S, row_off + rl, c) : 0.f;
  }
  __syncthreads();
  float mx = 0.f;
  for (int rr = ty; rr < 32; rr += 8) {
    const int rl = rb + rr, c = cb + tx;
    float w = 0.f;
    if (rl < nrows && c < R) {
      const int r = row_off + rl;
      w = (c == r) ? 0.f : w_direct(S, r, c) + tt[tx][rr];
      Wtmp[(long long)rl * Rp + c] = w;
    }
    mx = fmaxf(mx, fabsf(w));
    const float sum = warp_sum(w);
    if (tx == 0 && rl < nrows) rs_part[(long long)blockIdx.x * nrows + rl] = sum;
  }
  mx = warp_max(mx);
  if (tx == 0 && mx > 0.f && mx < 3.0e38f) atomicMax(wabs, __float_as_uint(mx));
}

__global__ void __launch_bounds__(256) w_rowsum_kernel(const float* __restrict__ rs_part, int nct, int nrows,
                                                       float* __restrict__ rowsum, unsigned* __restrict__ dabs) {
  const int r = blockIdx.x * 256 + threadIdx.x;
  float acc = 0.f;
  if (r < nrows) {
    for (int ct = 0; ct < nct; ++ct) acc += rs_part[(long long)ct * nrows + r];
    rowsum[r] = acc;
  }
  const float mx = warp_max(fabsf(acc));
  if ((threadIdx.x & 31) == 0 && mx > 0.f && mx < 3.0e38f) atomicMax(dabs, __float_as_uint(mx));
}

// grid (ceil(R / 256), nrows)
__global__ void __launch_bounds__(256) w_convert_kernel(const float* __restrict__ Wtmp, const float* __restrict__ rowsum,
                                                        float* __restrict__ scal, int row_off, int R, int Rp,
                                                        __half* __restrict__ Wh1, __half* __restrict__ Wh2) {
  const unsigned* sb = reinterpret_cast<const unsigned*>(scal);
  const unsigned bits = max(sb[kScalWabs], sb[kScalDabs]);
  const int e = bits ? 13 - floor_log2_bits(bits) : 0;       // max |W'| < 2^(ex + 1)  ->  < 2^14 after scaling
  const float ws = pow2f(e);
  const int rl = blockIdx.y, c = blockIdx.x * 256 + threadIdx.x;
  if (c < R) {
    const float w = (c == row_off + rl) ? -rowsum[rl] : Wtmp[(long long)rl * Rp + c];
    const float v = w * ws;
    const __half h1 = __float2half_rn(v);
    Wh1[(long long)rl * Rp + c] = h1;
    Wh2[(long long)rl * Rp + c] = __float2half_rn(v - __half2float(h1));
  }
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) scal[kScalGradAlpha] = pow2f(-e) * scal[kScalZinv];
}

// ---- shared context frames (row shards) ------------------------------------------------------------
// Column c of the video rows is a CONTEXT column when c % period < clen: x (real) and y (fake) hold the same values
// there, so y's are never read and x's stand in for them.  The split writes the columns permuted (the Gram and the
// row norms do not depend on the column order): the nc context columns first, zero-padded to Kcp (a multiple of 64),
// then the nq predicted columns, zero-padded as well.  K < 2^31 (checked by the callers): 32-bit column arithmetic.
__device__ __forceinline__ float ld_video(const float* __restrict__ p, long long i) { return p[i]; }
__device__ __forceinline__ float ld_video(const uint16_t* __restrict__ p, long long i) { return ld1(p, i); }
__device__ __forceinline__ float4 ld_video4(const float* __restrict__ p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ld_video4(const uint16_t* __restrict__ p) {
  return widen_bf16x4(*reinterpret_cast<const uint2*>(p));
}

// colsum_part_kernel with y's context columns read from x: the same sums, in the same order, on inputs that keep the
// promise
template <typename T>
__global__ void __launch_bounds__(128) colsum_part_ctx_kernel(const T* __restrict__ x, const T* __restrict__ y, int Bx,
                                                              int By, long long K, int period, int clen,
                                                              int rows_per_seg, float* __restrict__ part,
                                                              unsigned* __restrict__ absmax) {
  const long long k = (long long)blockIdx.x * 128 + threadIdx.x;
  const int R = Bx + By;
  const int r0 = blockIdx.y * rows_per_seg, r1 = min(R, r0 + rows_per_seg);
  float acc = 0.f, mx = 0.f;
  if (k < K) {
    const T* yk = ((int)k % period < clen) ? x : y;
    int r = r0;
    for (; r + 4 <= r1; r += 4) {
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int rr = r + u;
        v[u] = (rr < Bx) ? ld_video(x, (long long)rr * K + k) : ld_video(yk, (long long)(rr - Bx) * K + k);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) { acc += v[u]; mx = fmaxf(mx, fabsf(v[u])); }
    }
    for (; r < r1; ++r) {
      const float v = (r < Bx) ? ld_video(x, (long long)r * K + k) : ld_video(yk, (long long)(r - Bx) * K + k);
      acc += v;
      mx = fmaxf(mx, fabsf(v));
    }
    part[(long long)blockIdx.y * K + k] = acc;
  }
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0 && mx > 0.f && mx < 3.0e38f) atomicMax(absmax, __float_as_uint(mx));
}

// video column of permuted column j, or -1 for a padding column
__device__ __forceinline__ int ctx_source_col(int j, int period, int clen, int nc, int nq, int Kcp) {
  if (j < Kcp) return j < nc ? (j / clen) * period + j % clen : -1;
  j -= Kcp;
  const int pl = period - clen;
  return j < nq ? (j / pl) * period + clen + j % pl : -1;
}

// split_kernel over the permuted columns: grid (Kpp / 64, ceil(R / 64)), Zh [R][Kpp], ZT [Kpp][Rp].  A 64-column tile
// lies wholly in the context part or wholly in the predicted part (Kcp is a multiple of 64).
template <typename T>
__global__ void __launch_bounds__(256) split_ctx_kernel(const T* __restrict__ x, const T* __restrict__ y, int Bx, int By,
                                                        long long K, int period, int clen, int Kcp, long long Kpp,
                                                        int Rp, const float* __restrict__ mean,
                                                        const float* __restrict__ scal, __half* __restrict__ Zh1,
                                                        __half* __restrict__ Zh2, __half* __restrict__ ZT1,
                                                        __half* __restrict__ ZT2) {
  __shared__ __half t1[64][72], t2[64][72];                 // [column][row] for the transposed copy
  const int R = Bx + By;
  const int nc = (int)(K / period) * clen, nq = (int)K - nc;
  const int c0 = blockIdx.x * 64;
  const int r0 = blockIdx.y * 64;
  const int t = threadIdx.x;
  const int cg = (t & 15) * 4;
  const float zs = scal[kScalZscale];
  const T* yt = c0 < Kcp ? x : y;                           // source of the fake rows in this tile
  int src[4];
  float m[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    src[e] = ctx_source_col(c0 + cg + e, period, clen, nc, nq, Kcp);
    m[e] = src[e] >= 0 ? mean[src[e]] : 0.f;
  }
  // four permuted columns are four consecutive video columns when both part lengths are multiples of 4
  const bool vec = ((clen & 3) == 0) && ((period & 3) == 0) && src[0] >= 0 &&
                   ((reinterpret_cast<uintptr_t>(x) & (4 * sizeof(T) - 1)) == 0) &&
                   ((reinterpret_cast<uintptr_t>(y) & (4 * sizeof(T) - 1)) == 0);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int rl = (t >> 4) + 16 * i;
    const int r = r0 + rl;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (r < R) {
      const T* row = (r < Bx) ? x + (long long)r * K : yt + (long long)(r - Bx) * K;
      if (vec) {
        const float4 q = ld_video4(row + src[0]);
        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (src[e] >= 0) v[e] = ld_video(row, src[e]);
      }
    }
    __half h1[4], h2[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const bool in = (r < R) && src[e] >= 0;
      const float z = in ? (v[e] - m[e]) * zs : 0.f;
      h1[e] = __float2half_rn(z);
      h2[e] = __float2half_rn(z - __half2float(h1[e]));
    }
    if (r < R) {
      *reinterpret_cast<uint2*>(Zh1 + (long long)r * Kpp + c0 + cg) = *reinterpret_cast<const uint2*>(h1);
      *reinterpret_cast<uint2*>(Zh2 + (long long)r * Kpp + c0 + cg) = *reinterpret_cast<const uint2*>(h2);
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) { t1[cg + e][rl] = h1[e]; t2[cg + e][rl] = h2[e]; }
  }
  __syncthreads();
  // transposed rows: 4 threads per column, 16 stacked rows (32 bytes) each
  const int c = t >> 2, seg = (t & 3) * 16;
  if (r0 + seg < Rp) {                                      // Rp is a multiple of 64
    const uint4* s1 = reinterpret_cast<const uint4*>(&t1[c][seg]);
    const uint4* s2 = reinterpret_cast<const uint4*>(&t2[c][seg]);
    uint4* d1 = reinterpret_cast<uint4*>(ZT1 + (c0 + c) * (long long)Rp + r0 + seg);
    uint4* d2 = reinterpret_cast<uint4*>(ZT2 + (c0 + c) * (long long)Rp + r0 + seg);
    d1[0] = s1[0]; d1[1] = s1[1];
    d2[0] = s2[0]; d2[1] = s2[1];
  }
}

// gradient rows of the predicted columns, g_pred [nrows][nq] (fp32 or bf16 bits), back to the video columns of
// g [nrows][K]; the context columns are written as zero.  grid (ceil(K / 256), nrows)
template <typename G>
__global__ void __launch_bounds__(256) ctx_scatter_kernel(const G* __restrict__ g_pred, int K, int period, int clen,
                                                          G* __restrict__ g) {
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= K) return;
  const int pl = period - clen, nq = K / period * pl;
  const int ph = c % period;
  const long long r = blockIdx.y;
  g[r * K + c] = ph < clen ? G(0) : g_pred[r * nq + (c / period) * pl + (ph - clen)];
}
}  // namespace

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
namespace {
// the pre-pass kernels of an input element type
template <typename T>
struct Prep;
template <>
struct Prep<float> {
  static constexpr auto colsum = colsum_part_kernel;
  static constexpr auto split = split_kernel;
};
template <>
struct Prep<uint16_t> {
  static constexpr auto colsum = colsum_part_bf16_kernel;
  static constexpr auto split = split_bf16_kernel;
};

template <typename T>
int launch_stats(const T* x, const T* y, int Bx, int By, long long K, int nseg, float* part, float* mean, float* scal,
                 cudaStream_t st) {
  const int R = Bx + By;
  const int rps = (R + nseg - 1) / nseg;
  KCCOT_CUDA(cudaMemsetAsync(scal, 0, kScalCount * sizeof(float), st));
  Prep<T>::colsum<<<dim3((unsigned)((K + 127) / 128), nseg), 128, 0, st>>>(
      x, y, Bx, By, K, rps, part, reinterpret_cast<unsigned*>(scal) + kScalAbsmax);
  KCCOT_LAUNCH_CHECK();
  colmean_kernel<<<(unsigned)((K + 255) / 256), 256, 0, st>>>(part, (R + rps - 1) / rps, K, R, mean, scal);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}

template <typename T>
int launch_split(const T* x, const T* y, int Bx, int By, long long K, long long Kp, int Rp, const float* mean,
                 const float* scal, __half* Zh1, __half* Zh2, __half* ZT1, __half* ZT2, cudaStream_t st) {
  const int R = Bx + By;
  Prep<T>::split<<<dim3((unsigned)((K + 63) / 64), (R + 63) / 64), 256, 0, st>>>(x, y, Bx, By, K, Kp, Rp, mean,
                                                                                        scal, Zh1, Zh2, ZT1, ZT2);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}
}  // namespace

int large_launch_stats(const float* x, const float* y, int Bx, int By, long long K, int nseg, float* part, float* mean,
                       float* scal, cudaStream_t st) {
  return launch_stats(x, y, Bx, By, K, nseg, part, mean, scal, st);
}
int large_launch_stats(const uint16_t* x, const uint16_t* y, int Bx, int By, long long K, int nseg, float* part,
                       float* mean, float* scal, cudaStream_t st) {
  return launch_stats(x, y, Bx, By, K, nseg, part, mean, scal, st);
}

int large_launch_split(const float* x, const float* y, int Bx, int By, long long K, long long Kp, int Rp,
                       const float* mean, const float* scal, __half* Zh1, __half* Zh2, __half* ZT1, __half* ZT2,
                       cudaStream_t st) {
  return launch_split(x, y, Bx, By, K, Kp, Rp, mean, scal, Zh1, Zh2, ZT1, ZT2, st);
}
int large_launch_split(const uint16_t* x, const uint16_t* y, int Bx, int By, long long K, long long Kp, int Rp,
                       const float* mean, const float* scal, __half* Zh1, __half* Zh2, __half* ZT1, __half* ZT2,
                       cudaStream_t st) {
  return launch_split(x, y, Bx, By, K, Kp, Rp, mean, scal, Zh1, Zh2, ZT1, ZT2, st);
}

namespace {
template <typename T>
int launch_stats_ctx(const T* x, const T* y, int B, long long K, int period, int clen, int nseg, float* part, float* mean,
                     float* scal, cudaStream_t st) {
  const int R = 2 * B;
  const int rps = (R + nseg - 1) / nseg;
  KCCOT_CUDA(cudaMemsetAsync(scal, 0, kScalCount * sizeof(float), st));
  colsum_part_ctx_kernel<T><<<dim3((unsigned)((K + 127) / 128), nseg), 128, 0, st>>>(
      x, y, B, B, K, period, clen, rps, part, reinterpret_cast<unsigned*>(scal) + kScalAbsmax);
  KCCOT_LAUNCH_CHECK();
  colmean_kernel<<<(unsigned)((K + 255) / 256), 256, 0, st>>>(part, (R + rps - 1) / rps, K, R, mean, scal);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}

template <typename T>
int launch_split_ctx(const T* x, const T* y, int B, long long K, int period, int clen, int Kcp, long long Kpp, int Rp,
                     const float* mean, const float* scal, __half* Zh1, __half* Zh2, __half* ZT1, __half* ZT2,
                     cudaStream_t st) {
  split_ctx_kernel<T><<<dim3((unsigned)(Kpp / 64), (2 * B + 63) / 64), 256, 0, st>>>(
      x, y, B, B, K, period, clen, Kcp, Kpp, Rp, mean, scal, Zh1, Zh2, ZT1, ZT2);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}

template <typename G>
int launch_ctx_scatter(const G* g_pred, int nrows, int K, int period, int clen, G* g, cudaStream_t st) {
  ctx_scatter_kernel<G><<<dim3((unsigned)((K + 255) / 256), nrows), 256, 0, st>>>(g_pred, K, period, clen, g);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}
}  // namespace

int large_launch_stats_ctx(const float* x, const float* y, int B, long long K, int period, int clen, int nseg,
                           float* part, float* mean, float* scal, cudaStream_t st) {
  return launch_stats_ctx(x, y, B, K, period, clen, nseg, part, mean, scal, st);
}
int large_launch_stats_ctx(const uint16_t* x, const uint16_t* y, int B, long long K, int period, int clen, int nseg,
                           float* part, float* mean, float* scal, cudaStream_t st) {
  return launch_stats_ctx(x, y, B, K, period, clen, nseg, part, mean, scal, st);
}
int large_launch_split_ctx(const float* x, const float* y, int B, long long K, int period, int clen, int Kcp,
                           long long Kpp, int Rp, const float* mean, const float* scal, __half* Zh1, __half* Zh2,
                           __half* ZT1, __half* ZT2, cudaStream_t st) {
  return launch_split_ctx(x, y, B, K, period, clen, Kcp, Kpp, Rp, mean, scal, Zh1, Zh2, ZT1, ZT2, st);
}
int large_launch_split_ctx(const uint16_t* x, const uint16_t* y, int B, long long K, int period, int clen, int Kcp,
                           long long Kpp, int Rp, const float* mean, const float* scal, __half* Zh1, __half* Zh2,
                           __half* ZT1, __half* ZT2, cudaStream_t st) {
  return launch_split_ctx(x, y, B, K, period, clen, Kcp, Kpp, Rp, mean, scal, Zh1, Zh2, ZT1, ZT2, st);
}
int large_launch_ctx_scatter(const float* g_pred, int nrows, int K, int period, int clen, float* g, cudaStream_t st) {
  return launch_ctx_scatter(g_pred, nrows, K, period, clen, g, st);
}
int large_launch_ctx_scatter(const uint16_t* g_pred, int nrows, int K, int period, int clen, uint16_t* g,
                             cudaStream_t st) {
  return launch_ctx_scatter(g_pred, nrows, K, period, clen, g, st);
}

int large_launch_rownorm(const __half* Zh1, const __half* Zh2, int R, long long K, long long Kp, float* norms,
                         cudaStream_t st) {
  rownorm_kernel<<<R, 256, 0, st>>>(Zh1, Zh2, K, Kp, norms);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}

int large_launch_finalize(const LargeFin& F, int nblocks, int T, int J, float s, const float* scal, cudaStream_t st) {
  int mx = 0, my = 0;
  for (int q = 0; q < nblocks; ++q) {
    mx = max(mx, F.b[q].Bx);
    my = max(my, F.b[q].By);
  }
  large_finalize_kernel<<<dim3((my + 63) / 64, (mx + 63) / 64, nblocks), 256, 0, st>>>(F, T, J, s, scal);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}

int large_launch_wbuild(const float* Cxx, const float* Cxy, const float* Cyy, int Bx, int By, int row_off, int nrows,
                        int Rp, float* Wtmp, float* rs_part, float* rowsum, float* scal, __half* Wh1, __half* Wh2,
                        cudaStream_t st) {
  const int R = Bx + By;
  const int nct = (R + 31) / 32;
  WSrc S{Cxx, Cxy, Cyy, Bx, By, nullptr, nullptr, nullptr, 0, 0};
  unsigned* sb = reinterpret_cast<unsigned*>(scal);
  KCCOT_CUDA(cudaMemsetAsync(sb + kScalWabs, 0, 2 * sizeof(unsigned), st));
  w_tiles_kernel<<<dim3(nct, (nrows + 31) / 32), dim3(32, 8), 0, st>>>(S, row_off, nrows, Rp, Wtmp, rs_part, sb + kScalWabs);
  KCCOT_LAUNCH_CHECK();
  w_rowsum_kernel<<<(nrows + 255) / 256, 256, 0, st>>>(rs_part, nct, nrows, rowsum, sb + kScalDabs);
  KCCOT_LAUNCH_CHECK();
  w_convert_kernel<<<dim3((R + 255) / 256, nrows), 256, 0, st>>>(Wtmp, rowsum, scal, row_off, R, Rp, Wh1, Wh2);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}

int large_launch_wbuild_shard(const float* XYcol, const float* YYcol, const float* YYrow, int Bx, int By, int row0, int nloc,
                              int Rp, float* Wtmp, float* rs_part, float* rowsum, float* scal, __half* Wh1, __half* Wh2,
                              cudaStream_t st) {
  const int R = Bx + By;
  const int nct = (R + 31) / 32;
  const int row_off = Bx + row0;                       // stacked index of the first wanted row
  WSrc S{nullptr, nullptr, nullptr, Bx, By, XYcol, YYcol, YYrow, row0, nloc};
  unsigned* sb = reinterpret_cast<unsigned*>(scal);
  KCCOT_CUDA(cudaMemsetAsync(sb + kScalWabs, 0, 2 * sizeof(unsigned), st));
  w_tiles_kernel<<<dim3(nct, (nloc + 31) / 32), dim3(32, 8), 0, st>>>(S, row_off, nloc, Rp, Wtmp, rs_part, sb + kScalWabs);
  KCCOT_LAUNCH_CHECK();
  w_rowsum_kernel<<<(nloc + 255) / 256, 256, 0, st>>>(rs_part, nct, nloc, rowsum, sb + kScalDabs);
  KCCOT_LAUNCH_CHECK();
  w_convert_kernel<<<dim3((R + 255) / 256, nloc), 256, 0, st>>>(Wtmp, rowsum, scal, row_off, R, Rp, Wh1, Wh2);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}

}  // namespace kccot
