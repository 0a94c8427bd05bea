// Gaussian kernel smoothing of [B,H,T,W,C] videos (data_utils.py:503-521 temporal_convolution,
// :552-582 gaussian_convolution3D): separable REFLECT-padded 7-tap passes along T (mode 1) or
// H, T, W (mode 3), then division by the global maximum of the filtered tensor.
//
// A pass views the tensor as [outer, n, inner] and applies out[o,p,i] = sum_q A[p,q] in[o,q,i], with A the
// [n,n] matrix of the REFLECT-padded filter: A[p][reflect(p + k - R)] += w[k].  The 2R+1 weights travel as KERNEL
// ARGUMENTS (no filter matrix in device memory, no host-to-device copy when sigma is annealed every step,
// data_utils.py:584-586); each kernel derives the band coefficients it needs.  A (and its transpose, the
// adjoint) is banded with radius R, so every output row needs the rows p-R..p+R and 2R+1 coefficients
// coef[p][d].  R = 1..6 (kernel sizes 2..13; kernel_train.py:216 uses 6 -> R = 3, the class default 8 -> R = 4).
// Two kernels, neither with index arithmetic in its inner loop:
//   axis_col_kernel  (inner >= 64 or n*inner > 1024): one thread per (o, 4 consecutive inner elements) walks
//                    the n rows with a 7-row register window — every input element is loaded once, 16 bytes
//                    at a time, coalesced along `inner`;
//   axis_tile_kernel (small inner, e.g. the W pass with inner = C): a CTA copies a contiguous block of
//                    o_chunk * n * inner floats to shared memory, thread t = (p, i) keeps its 7 coefficients
//                    and row offsets in registers and produces out[o][p][i] for every o of the block.
// (The first version used one generic tile kernel with three integer divisions per element: 190 us for a
//  37.7 MB tensor, 20x off the HBM roofline.)
#include <type_traits>

#include "common.cuh"

namespace kccot {
namespace {
constexpr int FT = 256;
constexpr int kTileElems = 8192;     // 32 KB of shared memory per tile
constexpr int kMaxRadius = 6;
constexpr int kMaxAxis = 1024;       // coefficient table: n * (2R+1) floats of dynamic shared memory

struct Taps {                        // by value in the kernel parameters
  float w[2 * kMaxRadius + 1];
  int r;
};
__device__ __forceinline__ int reflect(int q, int n) { return q < 0 ? -q : (q >= n ? 2 * (n - 1) - q : q); }
// the 2R+1 weights of a pass: the kernel arguments, or, when wdev is set (the *_dev entries), device memory read as
// the kernel starts, so that a replayed CUDA graph filters with the buffer's current values.  (These kernels use no
// programmatic dependent launch; one that did would have to read wdev after griddepcontrol.wait.)
template <int R>
__device__ __forceinline__ void load_weights(float (&w)[2 * R + 1], const Taps& tp, const float* wdev) {
#pragma unroll
  for (int k = 0; k < 2 * R + 1; ++k) w[k] = wdev != nullptr ? wdev[k] : tp.w[k];
}
// A[p][q] of the REFLECT-padded filter (or its transpose)
template <int R>
__device__ __forceinline__ float band_coef(const float (&w)[2 * R + 1], int n, int p, int q, bool transposed) {
  const int row = transposed ? q : p, col = transposed ? p : q;
  float a = 0.f;
#pragma unroll
  for (int k = 0; k < 2 * R + 1; ++k) a += (reflect(row + k - R, n) == col) ? w[k] : 0.f;
  return a;
}

__device__ __forceinline__ void atomic_max_float(float* addr, float v) {
  if (v >= 0.f) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMin(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

struct BwdIn {            // input transform of the first adjoint pass: gz = gout/m + tie * (-S/m) / count
  const float* out;       // forward output (== 1.0f exactly where the max was attained)
  const float* maxval;
  const float* sums;      // [0] = sum(gout*out), [1] = number of tied maxima
};

template <int V> struct Vec;
template <> struct Vec<4> {
  float4 v;
  __device__ __forceinline__ void zero() { v = make_float4(0.f, 0.f, 0.f, 0.f); }
  __device__ __forceinline__ void load(const float* p) { v = *reinterpret_cast<const float4*>(p); }
  __device__ __forceinline__ void store(float* p) const { *reinterpret_cast<float4*>(p) = v; }
  __device__ __forceinline__ void fma(float c, const Vec& o) {
    v.x = fmaf(c, o.v.x, v.x); v.y = fmaf(c, o.v.y, v.y); v.z = fmaf(c, o.v.z, v.z); v.w = fmaf(c, o.v.w, v.w);
  }
  __device__ __forceinline__ void div(float d) { v.x /= d; v.y /= d; v.z /= d; v.w /= d; }
  __device__ __forceinline__ float hmax() const { return fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)); }
  __device__ __forceinline__ void bwd(float sc, float tie, const float* o) {
    const float4 t = *reinterpret_cast<const float4*>(o);
    v.x = v.x * sc + ((t.x == 1.0f) ? tie : 0.f); v.y = v.y * sc + ((t.y == 1.0f) ? tie : 0.f);
    v.z = v.z * sc + ((t.z == 1.0f) ? tie : 0.f); v.w = v.w * sc + ((t.w == 1.0f) ? tie : 0.f);
  }
};
template <> struct Vec<1> {
  float v;
  __device__ __forceinline__ void zero() { v = 0.f; }
  __device__ __forceinline__ void load(const float* p) { v = *p; }
  __device__ __forceinline__ void store(float* p) const { *p = v; }
  __device__ __forceinline__ void fma(float c, const Vec& o) { v = fmaf(c, o.v, v); }
  __device__ __forceinline__ void div(float d) { v /= d; }
  __device__ __forceinline__ float hmax() const { return v; }
  __device__ __forceinline__ void bwd(float sc, float tie, const float* o) { v = v * sc + ((*o == 1.0f) ? tie : 0.f); }
};

// MODE bit 0: write `out`; bit 1: reduce the global max into *gmax; bit 2: divide by *divisor;
// bit 3: apply the BwdIn transform on load; bit 4: use A transposed
template <int MODE, int V, int R>
__global__ void __launch_bounds__(FT) axis_col_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                      long long outer, int n, long long inner,
                                                      const Taps tp, const float* wdev, float* gmax,
                                                      const float* divisor, BwdIn bw) {
  constexpr int kR = R, kTaps = 2 * R + 1;
  extern __shared__ float coef[];                          // coef[p][d] = A[p][p + d - R] (0 outside the matrix)
  float w[kTaps];
  load_weights<R>(w, tp, wdev);
  for (int e = threadIdx.x; e < n * kTaps; e += FT) {
    const int p = e / kTaps, q = p + (e % kTaps) - kR;
    coef[e] = (q >= 0 && q < n) ? band_coef<R>(w, n, p, q, (MODE & 16) != 0) : 0.f;
  }
  __syncthreads();
  const long long iv = inner / V;
  const long long gid = (long long)blockIdx.x * FT + threadIdx.x;
  float lmax = -3.0e38f;
  if (gid < outer * iv) {
    const long long o = gid / iv;
    const long long base = o * n * inner + (gid - o * iv) * V;
    float gscale = 0.f, gtie = 0.f, inv = 1.f;
    if (MODE & 8) {
      const float m = *bw.maxval;
      gscale = 1.f / m;
      gtie = -(bw.sums[0] / m) / bw.sums[1];
    }
    if (MODE & 4) inv = *divisor;
    auto fetch = [&](int q) {
      Vec<V> r;
      if (q < n) {
        r.load(in + base + (long long)q * inner);
        if (MODE & 8) r.bwd(gscale, gtie, bw.out + base + (long long)q * inner);
      } else {
        r.zero();
      }
      return r;
    };
    Vec<V> win[kTaps];                                     // rows p-3 .. p+3
#pragma unroll
    for (int d = 0; d < kR; ++d) win[d].zero();
#pragma unroll
    for (int d = kR; d < kTaps; ++d) win[d] = fetch(d - kR);
    for (int p = 0; p < n; ++p) {
      const Vec<V> next = fetch(p + kR + 1);              // issued before the arithmetic of this row
      Vec<V> acc;
      acc.zero();
#pragma unroll
      for (int d = 0; d < kTaps; ++d) acc.fma(coef[p * kTaps + d], win[d]);
      if (MODE & 4) acc.div(inv);
      if (MODE & 2) lmax = fmaxf(lmax, acc.hmax());
      if (MODE & 1) acc.store(out + base + (long long)p * inner);
#pragma unroll
      for (int d = 0; d < kTaps - 1; ++d) win[d] = win[d + 1];
      win[kTaps - 1] = next;
    }
  }
  if (MODE & 2) {
    lmax = warp_max(lmax);
    if ((threadIdx.x & 31) == 0) atomic_max_float(gmax, lmax);
  }
}

template <int MODE, int R>
__global__ void __launch_bounds__(1024) axis_tile_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                         long long outer, int n, int inner, int o_chunk,
                                                         const Taps tp, const float* wdev, float* gmax,
                                                         const float* divisor, BwdIn bw) {
  constexpr int kR = R, kTaps = 2 * R + 1;
  extern __shared__ __align__(16) float tile[];            // [o_chunk][n][inner], contiguous like global memory
  const int ni = n * inner;
  const long long o0 = (long long)blockIdx.x * o_chunk;
  const int no = (int)min((long long)o_chunk, outer - o0);
  const long long g0 = o0 * ni;
  const int telems = no * ni;
  float gscale = 0.f, gtie = 0.f, inv = 1.f;
  if (MODE & 8) {
    const float m = *bw.maxval;
    gscale = 1.f / m;
    gtie = -(bw.sums[0] / m) / bw.sums[1];
  }
  if (MODE & 4) inv = *divisor;
  if ((ni & 3) == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0 &&
      (!(MODE & 8) || (reinterpret_cast<uintptr_t>(bw.out) & 15) == 0)) {
    for (int e = threadIdx.x * 4; e < telems; e += blockDim.x * 4) {
      Vec<4> r;
      r.load(in + g0 + e);
      if (MODE & 8) r.bwd(gscale, gtie, bw.out + g0 + e);
      r.store(tile + e);
    }
  } else {
    for (int e = threadIdx.x; e < telems; e += blockDim.x) {
      Vec<1> r;
      r.load(in + g0 + e);
      if (MODE & 8) r.bwd(gscale, gtie, bw.out + g0 + e);
      tile[e] = r.v;
    }
  }
  // thread t = (p, i): its 7 coefficients and (clamped) row offsets stay in registers
  const int t = threadIdx.x;
  float c[kTaps];
  int off[kTaps];
  {
    const int p = min(t, ni - 1) / inner;
    float w[kTaps];
    load_weights<R>(w, tp, wdev);
#pragma unroll
    for (int d = 0; d < kTaps; ++d) {
      const int q = p + d - kR;
      const bool ok = q >= 0 && q < n;
      c[d] = ok ? band_coef<R>(w, n, p, q, (MODE & 16) != 0) : 0.f;
      off[d] = ok ? (d - kR) * inner : 0;
    }
  }
  __syncthreads();
  float lmax = -3.0e38f;
  if (t < ni) {
    for (int oo = 0; oo < no; ++oo) {
      const float* row = tile + oo * ni + t;
      float acc = 0.f;
#pragma unroll
      for (int d = 0; d < kTaps; ++d) acc = fmaf(c[d], row[off[d]], acc);
      if (MODE & 4) acc = acc / inv;
      if (MODE & 2) lmax = fmaxf(lmax, acc);
      if (MODE & 1) out[g0 + (long long)oo * ni + t] = acc;
    }
  }
  if (MODE & 2) {
    lmax = warp_max(lmax);
    if ((threadIdx.x & 31) == 0) atomic_max_float(gmax, lmax);
  }
}

__global__ void init_max_kernel(float* m) { *m = __int_as_float(0xff800000); }

// sums[0] = sum gout * out, sums[1] = number of elements at the maximum (out == 1).  16-byte loads, four in flight per
// thread (the scalar grid-stride version ran at 2.5 TB/s: 29.9 us for the 75.5 MB of config 3).
__global__ void __launch_bounds__(FT) tie_sums_kernel(const float* __restrict__ gout, const float* __restrict__ out,
                                                      long long n, float* sums) {
  float s = 0.f, c = 0.f;
  const long long stride = (long long)gridDim.x * FT;
  const long long tid = (long long)blockIdx.x * FT + threadIdx.x;
  const bool vec = ((reinterpret_cast<uintptr_t>(gout) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  const long long n4 = vec ? n / 4 : 0;
  const float4* g4 = reinterpret_cast<const float4*>(gout);
  const float4* o4 = reinterpret_cast<const float4*>(out);
  auto acc4 = [&](const float4& g, const float4& o) {
    s = fmaf(g.x, o.x, s); s = fmaf(g.y, o.y, s); s = fmaf(g.z, o.z, s); s = fmaf(g.w, o.w, s);
    c += (o.x == 1.0f ? 1.f : 0.f) + (o.y == 1.0f ? 1.f : 0.f) + (o.z == 1.0f ? 1.f : 0.f) + (o.w == 1.0f ? 1.f : 0.f);
  };
  long long i = tid;
  for (; i + 3 * stride < n4; i += 4 * stride) {
    float4 g[4], o[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { g[u] = __ldg(g4 + i + u * stride); o[u] = __ldg(o4 + i + u * stride); }
#pragma unroll
    for (int u = 0; u < 4; ++u) acc4(g[u], o[u]);
  }
  for (; i < n4; i += stride) acc4(__ldg(g4 + i), __ldg(o4 + i));
  for (long long k = 4 * n4 + tid; k < n; k += stride) {
    const float o = out[k];
    s = fmaf(gout[k], o, s);
    c += (o == 1.0f) ? 1.f : 0.f;
  }
  // one atomic pair per CTA: same-address atomics retire one at a time (19 000 of them were the kernel: 40 us)
  __shared__ float red[2][FT / 32];
  s = warp_sum(s);
  c = warp_sum(c);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s; red[1][threadIdx.x >> 5] = c; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float ss = 0.f, cc = 0.f;
#pragma unroll
    for (int w = 0; w < FT / 32; ++w) { ss += red[0][w]; cc += red[1][w]; }
    atomicAdd(&sums[0], ss);
    atomicAdd(&sums[1], cc);
  }
}

// ---- bf16 videos ----------------------------------------------------------------------------------------------------
// The bf16 passes are axis_col_kernel / axis_tile_kernel / tie_sums_kernel with other load and store sides, written as
// kernels of their own so that the fp32 kernels keep their code.  TI / TO is the element type a pass reads / writes:
// uint16_t (bf16 raw bits) on the first pass of a call and the last, float for the fp32 intermediates of mode 3, whose
// middle passes are the fp32 kernels themselves.  Loads widen (exact), every sum is formed in fp32 with the same
// coefficients and the same FMA order per element, whatever the vector width, and only the final store rounds (nearest
// even): the output is the fp32 call's output rounded.
// The backward needs the set of tied maxima, out == 1.0f in fp32, which a bf16 output cannot carry (every fp32 value in
// [1 - 2^-9, 1) rounds to 1.0).  So the forward's last pass sets bit e of `ties` where its fp32 quotient is exactly 1.0f
// (an atomicOr per tied element, so about one per call), and the backward reads the bit.
struct Ties {
  uint32_t* bits;         // bit e % 32 of bits[e / 32]: element e is a tied maximum.  Set by the forward's last pass
                          // (MODE & 4), read by the backward's first (MODE & 8)
  const float* maxval;
  const float* sums;      // [0] = sum(gout*out) over the bf16 out, [1] = number of tied maxima (popcount of bits)
};

// V = 8 (16-byte bf16 / 2 x 16-byte fp32 accesses), 4 (8-byte bf16 / 16-byte fp32 accesses) or 1
template <int V> struct VecF { float v[V]; };
template <int V, typename T>
__device__ __forceinline__ void load_v(VecF<V>& r, const T* p) {
  if constexpr (V == 8 && sizeof(T) == 2) {
    const uint4 u = *reinterpret_cast<const uint4*>(p);
    const float4 a = widen_bf16x4(make_uint2(u.x, u.y)), b = widen_bf16x4(make_uint2(u.z, u.w));
    r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w; r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
  } else if constexpr (V == 8) {
    const float4 a = reinterpret_cast<const float4*>(p)[0], b = reinterpret_cast<const float4*>(p)[1];
    r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w; r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
  } else if constexpr (V == 4) {
    const float4 a = sizeof(T) == 2 ? widen_bf16x4(*reinterpret_cast<const uint2*>(p))
                                    : *reinterpret_cast<const float4*>(p);
    r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
  } else if constexpr (sizeof(T) == 2) {
    r.v[0] = __uint_as_float((uint32_t)*p << 16);
  } else {
    r.v[0] = *p;
  }
}
template <int V, typename T>
__device__ __forceinline__ void store_v(T* p, const VecF<V>& r) {
  if constexpr (V == 8 && sizeof(T) == 2) {
    *reinterpret_cast<uint4*>(p) = make_uint4(pack_bf16x2(r.v[0], r.v[1]), pack_bf16x2(r.v[2], r.v[3]),
                                              pack_bf16x2(r.v[4], r.v[5]), pack_bf16x2(r.v[6], r.v[7]));
  } else if constexpr (V == 8) {
    reinterpret_cast<float4*>(p)[0] = make_float4(r.v[0], r.v[1], r.v[2], r.v[3]);
    reinterpret_cast<float4*>(p)[1] = make_float4(r.v[4], r.v[5], r.v[6], r.v[7]);
  } else if constexpr (V == 4 && sizeof(T) == 2) {
    *reinterpret_cast<uint2*>(p) = make_uint2(pack_bf16x2(r.v[0], r.v[1]), pack_bf16x2(r.v[2], r.v[3]));
  } else if constexpr (V == 4) {
    *reinterpret_cast<float4*>(p) = make_float4(r.v[0], r.v[1], r.v[2], r.v[3]);
  } else if constexpr (sizeof(T) == 2) {
    *p = __bfloat16_as_ushort(__float2bfloat16_rn(r.v[0]));
  } else {
    *p = r.v[0];
  }
}
// the BwdIn transform of the fp32 kernels with the tie bits in place of out == 1.0f; e % V == 0
template <int V>
__device__ __forceinline__ void bwd_v(VecF<V>& r, float sc, float tie, const uint32_t* bits, long long e) {
  const uint32_t b = bits[e >> 5] >> (e & 31);
#pragma unroll
  for (int j = 0; j < V; ++j) r.v[j] = r.v[j] * sc + (((b >> j) & 1u) ? tie : 0.f);
}
// sets the tie bits of the V elements e.. whose quotient is exactly 1.0f; e % V == 0
template <int V>
__device__ __forceinline__ void mark_ties(uint32_t* bits, const VecF<V>& r, long long e) {
  uint32_t b = 0;
#pragma unroll
  for (int j = 0; j < V; ++j) b |= (r.v[j] == 1.0f ? 1u : 0u) << j;
  if (b) atomicOr(bits + (e >> 5), b << (e & 31));
}

// axis_col_kernel for bf16 (MODE bits as there; MODE & 4 also marks the ties, MODE & 8 reads them)
template <typename TI, typename TO, int MODE, int V, int R>
__global__ void __launch_bounds__(FT) axis_col_bf16_kernel(const TI* __restrict__ in, TO* __restrict__ out,
                                                           long long outer, int n, long long inner, const Taps tp,
                                                           const float* wdev, float* gmax, const float* divisor,
                                                           Ties tie) {
  constexpr int kR = R, kTaps = 2 * R + 1;
  extern __shared__ float coef[];                          // coef[p][d] = A[p][p + d - R] (0 outside the matrix)
  float w[kTaps];
  load_weights<R>(w, tp, wdev);
  for (int e = threadIdx.x; e < n * kTaps; e += FT) {
    const int p = e / kTaps, q = p + (e % kTaps) - kR;
    coef[e] = (q >= 0 && q < n) ? band_coef<R>(w, n, p, q, (MODE & 16) != 0) : 0.f;
  }
  __syncthreads();
  const long long iv = inner / V;
  const long long gid = (long long)blockIdx.x * FT + threadIdx.x;
  float lmax = -3.0e38f;
  if (gid < outer * iv) {
    const long long o = gid / iv;
    const long long base = o * n * inner + (gid - o * iv) * V;
    float gscale = 0.f, gtie = 0.f, inv = 1.f;
    if (MODE & 8) {
      const float m = *tie.maxval;
      gscale = 1.f / m;
      gtie = -(tie.sums[0] / m) / tie.sums[1];
    }
    if (MODE & 4) inv = *divisor;
    auto fetch = [&](int q) {
      VecF<V> r;
      if (q < n) {
        load_v<V>(r, in + base + (long long)q * inner);
        if (MODE & 8) bwd_v<V>(r, gscale, gtie, tie.bits, base + (long long)q * inner);
      } else {
#pragma unroll
        for (int j = 0; j < V; ++j) r.v[j] = 0.f;
      }
      return r;
    };
    VecF<V> win[kTaps];
#pragma unroll
    for (int d = 0; d < kR; ++d)
#pragma unroll
      for (int j = 0; j < V; ++j) win[d].v[j] = 0.f;
#pragma unroll
    for (int d = kR; d < kTaps; ++d) win[d] = fetch(d - kR);
    // two rows in flight per thread where the window leaves registers for it (a bf16 pass has half the fp32 threads)
    constexpr bool kDeep = V * kTaps <= 64;
    VecF<V> next = fetch(kR + 1), next2;
    for (int p = 0; p < n; ++p) {
      if constexpr (kDeep) next2 = fetch(p + kR + 2);
      VecF<V> acc;
#pragma unroll
      for (int j = 0; j < V; ++j) acc.v[j] = 0.f;
#pragma unroll
      for (int d = 0; d < kTaps; ++d) {
        const float c = coef[p * kTaps + d];
#pragma unroll
        for (int j = 0; j < V; ++j) acc.v[j] = fmaf(c, win[d].v[j], acc.v[j]);
      }
      if (MODE & 4) {
#pragma unroll
        for (int j = 0; j < V; ++j) acc.v[j] /= inv;
        mark_ties<V>(tie.bits, acc, base + (long long)p * inner);
      }
      if (MODE & 2) {
#pragma unroll
        for (int j = 0; j < V; ++j) lmax = fmaxf(lmax, acc.v[j]);
      }
      if (MODE & 1) store_v<V>(out + base + (long long)p * inner, acc);
#pragma unroll
      for (int d = 0; d < kTaps - 1; ++d) win[d] = win[d + 1];
      win[kTaps - 1] = next;
      if constexpr (kDeep) next = next2;
      else next = fetch(p + kR + 2);
    }
  }
  if (MODE & 2) {
    lmax = warp_max(lmax);
    if ((threadIdx.x & 31) == 0) atomic_max_float(gmax, lmax);
  }
}

// axis_tile_kernel for bf16
template <typename TI, typename TO, int MODE, int R>
__global__ void __launch_bounds__(1024) axis_tile_bf16_kernel(const TI* __restrict__ in, TO* __restrict__ out,
                                                              long long outer, int n, int inner, int o_chunk,
                                                              const Taps tp, const float* wdev, float* gmax,
                                                              const float* divisor, Ties tie) {
  constexpr int kR = R, kTaps = 2 * R + 1;
  extern __shared__ __align__(16) float tile[];            // [o_chunk][n][inner], contiguous like global memory
  const int ni = n * inner;
  const long long o0 = (long long)blockIdx.x * o_chunk;
  const int no = (int)min((long long)o_chunk, outer - o0);
  const long long g0 = o0 * ni;
  const int telems = no * ni;
  float gscale = 0.f, gtie = 0.f, inv = 1.f;
  if (MODE & 8) {
    const float m = *tie.maxval;
    gscale = 1.f / m;
    gtie = -(tie.sums[0] / m) / tie.sums[1];
  }
  if (MODE & 4) inv = *divisor;
  if ((ni & 7) == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0) {
    for (int e = threadIdx.x * 8; e < telems; e += blockDim.x * 8) {
      VecF<8> r;
      load_v<8>(r, in + g0 + e);
      if (MODE & 8) bwd_v<8>(r, gscale, gtie, tie.bits, g0 + e);
      store_v<8>(tile + e, r);
    }
  } else {
    for (int e = threadIdx.x; e < telems; e += blockDim.x) {
      VecF<1> r;
      load_v<1>(r, in + g0 + e);
      if (MODE & 8) bwd_v<1>(r, gscale, gtie, tie.bits, g0 + e);
      tile[e] = r.v[0];
    }
  }
  const int t = threadIdx.x;
  float c[kTaps];
  int off[kTaps];
  {
    const int p = min(t, ni - 1) / inner;
    float w[kTaps];
    load_weights<R>(w, tp, wdev);
#pragma unroll
    for (int d = 0; d < kTaps; ++d) {
      const int q = p + d - kR;
      const bool ok = q >= 0 && q < n;
      c[d] = ok ? band_coef<R>(w, n, p, q, (MODE & 16) != 0) : 0.f;
      off[d] = ok ? (d - kR) * inner : 0;
    }
  }
  __syncthreads();
  float lmax = -3.0e38f;
  auto row_out = [&](int oo) {
    const float* row = tile + oo * ni + t;
    VecF<1> acc;
    acc.v[0] = 0.f;
#pragma unroll
    for (int d = 0; d < kTaps; ++d) acc.v[0] = fmaf(c[d], row[off[d]], acc.v[0]);
    const long long e = g0 + (long long)oo * ni + t;
    if (MODE & 4) {
      acc.v[0] = acc.v[0] / inv;
      mark_ties<1>(tie.bits, acc, e);
    }
    if (MODE & 2) lmax = fmaxf(lmax, acc.v[0]);
    if (MODE & 1) store_v<1>(out + e, acc);
  };
  if (t < ni) {
    if constexpr ((MODE & 2) != 0) {
#pragma unroll 1     // unrolled, the max pass spills at R = 5, 6 (64 registers per thread at 1024 threads)
      for (int oo = 0; oo < no; ++oo) row_out(oo);
    } else {
      for (int oo = 0; oo < no; ++oo) row_out(oo);
    }
  }
  if (MODE & 2) {
    lmax = warp_max(lmax);
    if ((threadIdx.x & 31) == 0) atomic_max_float(gmax, lmax);
  }
}

// tie_sums_kernel for bf16: sums[0] = sum gout * out (bf16 out), sums[1] = popcount of the tie bits (nwords words)
__global__ void __launch_bounds__(FT) tie_sums_bf16_kernel(const uint16_t* __restrict__ gout,
                                                           const uint16_t* __restrict__ out,
                                                           const uint32_t* __restrict__ bits, long long n,
                                                           long long nwords, float* sums) {
  float s = 0.f;
  unsigned cnt = 0;
  const long long stride = (long long)gridDim.x * FT;
  const long long tid = (long long)blockIdx.x * FT + threadIdx.x;
  const bool vec = ((reinterpret_cast<uintptr_t>(gout) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  const long long n8 = vec ? n / 8 : 0;
  const uint4* g8 = reinterpret_cast<const uint4*>(gout);
  const uint4* o8 = reinterpret_cast<const uint4*>(out);
  auto acc8 = [&](const uint4& g, const uint4& o) {
    const float4 g0 = widen_bf16x4(make_uint2(g.x, g.y)), g1 = widen_bf16x4(make_uint2(g.z, g.w));
    const float4 o0 = widen_bf16x4(make_uint2(o.x, o.y)), o1 = widen_bf16x4(make_uint2(o.z, o.w));
    s = fmaf(g0.x, o0.x, s); s = fmaf(g0.y, o0.y, s); s = fmaf(g0.z, o0.z, s); s = fmaf(g0.w, o0.w, s);
    s = fmaf(g1.x, o1.x, s); s = fmaf(g1.y, o1.y, s); s = fmaf(g1.z, o1.z, s); s = fmaf(g1.w, o1.w, s);
  };
  long long i = tid;
  for (; i + 3 * stride < n8; i += 4 * stride) {
    uint4 g[4], o[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { g[u] = __ldg(g8 + i + u * stride); o[u] = __ldg(o8 + i + u * stride); }
#pragma unroll
    for (int u = 0; u < 4; ++u) acc8(g[u], o[u]);
  }
  for (; i < n8; i += stride) acc8(__ldg(g8 + i), __ldg(o8 + i));
  for (long long k = 8 * n8 + tid; k < n; k += stride)
    s = fmaf(__uint_as_float((uint32_t)gout[k] << 16), __uint_as_float((uint32_t)out[k] << 16), s);
  for (long long w = tid; w < nwords; w += stride) cnt += __popc(bits[w]);
  __shared__ float red[2][FT / 32];
  s = warp_sum(s);
  const float c = warp_sum((float)cnt);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s; red[1][threadIdx.x >> 5] = c; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float ss = 0.f, cc = 0.f;
#pragma unroll
    for (int w = 0; w < FT / 32; ++w) { ss += red[0][w]; cc += red[1][w]; }
    atomicAdd(&sums[0], ss);
    atomicAdd(&sums[1], cc);
  }
}

struct AxisPlan { long long outer, inner; int n, o_chunk; bool tiled; };
AxisPlan plan_axis(long long outer, int n, long long inner) {
  AxisPlan p;
  p.outer = outer; p.inner = inner; p.n = n;
  p.tiled = (inner < 64) && ((long long)n * inner <= 1024);
  p.o_chunk = (int)max(1LL, (long long)kTileElems / ((long long)n * inner));
  return p;
}

template <int MODE, int R>
int run_axis_r(const float* in, float* out, const AxisPlan& p, const Taps& tp, const float* wdev, float* gmax,
               const float* divisor, BwdIn bw, cudaStream_t st) {
  if (p.tiled) {
    const int ni = p.n * (int)p.inner;
    const int threads = (ni + 31) / 32 * 32;
    const unsigned grid = (unsigned)((p.outer + p.o_chunk - 1) / p.o_chunk);
    const size_t smem = (size_t)p.o_chunk * ni * sizeof(float);
    axis_tile_kernel<MODE, R><<<grid, threads, smem, st>>>(in, out, p.outer, p.n, (int)p.inner, p.o_chunk, tp, wdev, gmax,
                                                           divisor, bw);
  } else {
    const bool v4 = (p.inner % 4 == 0) && (reinterpret_cast<uintptr_t>(in) & 15) == 0 &&
                    (!(MODE & 1) || (reinterpret_cast<uintptr_t>(out) & 15) == 0) &&
                    (!(MODE & 8) || (reinterpret_cast<uintptr_t>(bw.out) & 15) == 0);
    const long long total = p.outer * (p.inner / (v4 ? 4 : 1));
    const unsigned grid = (unsigned)((total + FT - 1) / FT);
    const size_t smem = (size_t)p.n * (2 * R + 1) * sizeof(float);       // <= 1024 * 13 * 4 = 52 KB
    if (smem > 48 * 1024) {
      if (v4) KCCOT_CUDA(cudaFuncSetAttribute(axis_col_kernel<MODE, 4, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      else KCCOT_CUDA(cudaFuncSetAttribute(axis_col_kernel<MODE, 1, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    if (v4) axis_col_kernel<MODE, 4, R><<<grid, FT, smem, st>>>(in, out, p.outer, p.n, p.inner, tp, wdev, gmax, divisor,
                                                                bw);
    else axis_col_kernel<MODE, 1, R><<<grid, FT, smem, st>>>(in, out, p.outer, p.n, p.inner, tp, wdev, gmax, divisor, bw);
  }
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}
template <int MODE>
int run_axis(const float* in, float* out, const AxisPlan& p, const Taps& tp, const float* wdev, float* gmax,
             const float* divisor, BwdIn bw, cudaStream_t st) {
  switch (tp.r) {
    case 1: return run_axis_r<MODE, 1>(in, out, p, tp, wdev, gmax, divisor, bw, st);
    case 2: return run_axis_r<MODE, 2>(in, out, p, tp, wdev, gmax, divisor, bw, st);
    case 3: return run_axis_r<MODE, 3>(in, out, p, tp, wdev, gmax, divisor, bw, st);
    case 4: return run_axis_r<MODE, 4>(in, out, p, tp, wdev, gmax, divisor, bw, st);
    case 5: return run_axis_r<MODE, 5>(in, out, p, tp, wdev, gmax, divisor, bw, st);
    case 6: return run_axis_r<MODE, 6>(in, out, p, tp, wdev, gmax, divisor, bw, st);
  }
  set_error("smoothing radius %d not supported (1..%d)", tp.r, kMaxRadius);
  return KCCOT_EUNSUPPORTED;
}
// w: host weights, copied into the kernel arguments, or (on_device) a device array the kernels read as wdev
int make_taps(Taps* tp, const float* w, int radius, const char* what, bool on_device = false) {
  KCCOT_CHECK_ARG(w != nullptr, "%s: null weights", what);
  KCCOT_CHECK_ARG(!on_device || (reinterpret_cast<uintptr_t>(w) & 3) == 0, "%s: device weights must be 4-byte aligned",
                  what);
  if (radius < 1 || radius > kMaxRadius) {
    set_error("%s: smoothing radius %d not supported (kernel sizes 2..%d, radius 1..%d)", what, radius, 2 * kMaxRadius + 1,
              kMaxRadius);
    return KCCOT_EUNSUPPORTED;
  }
  tp->r = radius;
  for (int k = 0; k < 2 * kMaxRadius + 1; ++k) tp->w[k] = !on_device && k < 2 * radius + 1 ? w[k] : 0.f;
  return KCCOT_OK;
}

// run_axis for the bf16 passes (TI / TO as in axis_col_bf16_kernel; MODE 2 passes write nothing and take TO = uint16_t)
template <typename TI, typename TO, int MODE, int R>
int run_axis_bf16_r(const TI* in, TO* out, const AxisPlan& p, const Taps& tp, const float* wdev, float* gmax,
                    const float* divisor, Ties tie, cudaStream_t st) {
  if (p.tiled) {
    const int ni = p.n * (int)p.inner;
    const int threads = (ni + 31) / 32 * 32;
    const unsigned grid = (unsigned)((p.outer + p.o_chunk - 1) / p.o_chunk);
    const size_t smem = (size_t)p.o_chunk * ni * sizeof(float);
    axis_tile_bf16_kernel<TI, TO, MODE, R><<<grid, threads, smem, st>>>(in, out, p.outer, p.n, (int)p.inner, p.o_chunk,
                                                                       tp, wdev, gmax, divisor, tie);
  } else {
    // widest access the shape and pointers allow, but 4 instead of 8 elements per thread while 8 would leave fewer
    // than ~1 000 threads per SM (config 3's T pass: 98 304 threads at 8, 196 608 at 4)
    auto fits = [&](int v) {
      const uintptr_t a = (uintptr_t)(v * sizeof(TI) < 16 ? v * sizeof(TI) : 16) - 1;
      const uintptr_t b = (uintptr_t)(v * sizeof(TO) < 16 ? v * sizeof(TO) : 16) - 1;
      return p.inner % v == 0 && (reinterpret_cast<uintptr_t>(in) & a) == 0 &&
             (!(MODE & 1) || (reinterpret_cast<uintptr_t>(out) & b) == 0);
    };
    const int v = fits(8) && p.outer * (p.inner / 8) >= 1024LL * num_sms() ? 8 : fits(4) ? 4 : fits(8) ? 8 : 1;
    const long long total = p.outer * (p.inner / v);
    const unsigned grid = (unsigned)((total + FT - 1) / FT);
    const size_t smem = (size_t)p.n * (2 * R + 1) * sizeof(float);
    auto kernel = v == 8 ? axis_col_bf16_kernel<TI, TO, MODE, 8, R>
                         : v == 4 ? axis_col_bf16_kernel<TI, TO, MODE, 4, R> : axis_col_bf16_kernel<TI, TO, MODE, 1, R>;
    if (smem > 48 * 1024)
      KCCOT_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<grid, FT, smem, st>>>(in, out, p.outer, p.n, p.inner, tp, wdev, gmax, divisor, tie);
  }
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}
template <typename TI, typename TO, int MODE>
int run_axis_bf16(const TI* in, TO* out, const AxisPlan& p, const Taps& tp, const float* wdev, float* gmax,
                  const float* divisor, Ties tie, cudaStream_t st) {
  switch (tp.r) {
    case 1: return run_axis_bf16_r<TI, TO, MODE, 1>(in, out, p, tp, wdev, gmax, divisor, tie, st);
    case 2: return run_axis_bf16_r<TI, TO, MODE, 2>(in, out, p, tp, wdev, gmax, divisor, tie, st);
    case 3: return run_axis_bf16_r<TI, TO, MODE, 3>(in, out, p, tp, wdev, gmax, divisor, tie, st);
    case 4: return run_axis_bf16_r<TI, TO, MODE, 4>(in, out, p, tp, wdev, gmax, divisor, tie, st);
    case 5: return run_axis_bf16_r<TI, TO, MODE, 5>(in, out, p, tp, wdev, gmax, divisor, tie, st);
    case 6: return run_axis_bf16_r<TI, TO, MODE, 6>(in, out, p, tp, wdev, gmax, divisor, tie, st);
  }
  set_error("smoothing radius %d not supported (1..%d)", tp.r, kMaxRadius);
  return KCCOT_EUNSUPPORTED;
}

// argument checks of the bf16 and the device-weight entries: those of kccot_smooth_fwd, all made before any CUDA call
int smooth_args(int mode, int B, int H, int T, int W, int C, const float* taps_t, int radius_t, const float* taps_s,
                int radius_s, bool taps_on_device, void* ws, size_t ws_bytes, Taps* tp) {
  KCCOT_CHECK_ARG(B >= 1 && H >= 1 && T >= 1 && W >= 1 && C >= 1, "bad sizes");
  KCCOT_CHECK_ARG(T <= kMaxAxis && H <= kMaxAxis && W <= kMaxAxis, "axis longer than %d not supported (H=%d T=%d W=%d)", kMaxAxis,
                  H, T, W);
  if (int rc = mode == 1 ? make_taps(tp, taps_t, radius_t, "temporal_convolution", taps_on_device)
                          : make_taps(tp, taps_s, radius_s, "gaussian_convolution3D", taps_on_device))
    return rc;
  KCCOT_CHECK_ARG(T > tp->r, "REFLECT padding by %d needs T > %d (T=%d)", tp->r, tp->r, T);
  if (mode == 3) {
    KCCOT_CHECK_ARG(H > tp->r && W > tp->r, "3-D smoothing needs H, W > %d (H=%d W=%d)", tp->r, H, W);
    KCCOT_CHECK_ARG(ws && ws_bytes >= kccot_smooth_workspace_bytes(mode, B, H, T, W, C), "workspace too small");
  }
  return KCCOT_OK;
}

// The passes of the four fp32 / bf16 entries, after their argument checks.  wdev == nullptr: the weights are tp.w
// (host arrays, the existing entries); otherwise the 2 * tp.r + 1 floats at wdev (the *_dev entries).
int smooth_fwd_f32(int mode, const float* x, int B, int H, int T, int W, int C, const Taps& tp, const float* wdev,
                   float* out, float* maxval, void* ws, size_t ws_bytes, cudaStream_t st) {
  init_max_kernel<<<1, 1, 0, st>>>(maxval);
  KCCOT_LAUNCH_CHECK();
  const AxisPlan pt = plan_axis((long long)B * H, T, (long long)W * C);
  BwdIn none{};
  if (mode == 1) {
    if (int rc = run_axis<2>(x, nullptr, pt, tp, wdev, maxval, nullptr, none, st)) return rc;
    return run_axis<1 | 4>(x, out, pt, tp, wdev, nullptr, maxval, none, st);
  }
  KCCOT_CHECK_ARG(H > tp.r && W > tp.r, "3-D smoothing needs H, W > %d (H=%d W=%d)", tp.r, H, W);
  const size_t n = align_up((size_t)B * H * T * W * C * sizeof(float), 256);
  KCCOT_CHECK_ARG(ws && ws_bytes >= 256 + 2 * n, "workspace too small");
  float* t1 = (float*)((char*)ws + 256);
  float* t2 = (float*)((char*)ws + 256 + n);
  const AxisPlan ph = plan_axis(B, H, (long long)T * W * C);
  const AxisPlan pw = plan_axis((long long)B * H * T, W, C);
  if (int rc = run_axis<1>(x, t1, ph, tp, wdev, nullptr, nullptr, none, st)) return rc;
  if (int rc = run_axis<1>(t1, t2, pt, tp, wdev, nullptr, nullptr, none, st)) return rc;
  if (int rc = run_axis<2>(t2, nullptr, pw, tp, wdev, maxval, nullptr, none, st)) return rc;
  return run_axis<1 | 4>(t2, out, pw, tp, wdev, nullptr, maxval, none, st);
}

int smooth_bwd_f32(int mode, const float* gout, const float* out, const float* maxval, int B, int H, int T, int W,
                   int C, const Taps& tp, const float* wdev, float* gx, void* ws, size_t ws_bytes, cudaStream_t st) {
  const long long nel = (long long)B * H * T * W * C;
  float* sums = (float*)ws;
  KCCOT_CUDA(cudaMemsetAsync(sums, 0, 2 * sizeof(float), st));
  tie_sums_kernel<<<(unsigned)min((long long)4 * num_sms(), (nel / 4 + FT - 1) / FT + 1), FT, 0, st>>>(gout, out, nel, sums);
  KCCOT_LAUNCH_CHECK();
  BwdIn bw{out, maxval, sums};
  BwdIn none{};
  const AxisPlan pt = plan_axis((long long)B * H, T, (long long)W * C);
  if (mode == 1) return run_axis<1 | 8 | 16>(gout, gx, pt, tp, wdev, nullptr, nullptr, bw, st);
  const size_t n = align_up((size_t)nel * sizeof(float), 256);
  KCCOT_CHECK_ARG(ws_bytes >= 256 + 2 * n, "workspace too small");
  float* t1 = (float*)((char*)ws + 256);
  float* t2 = (float*)((char*)ws + 256 + n);
  const AxisPlan ph = plan_axis(B, H, (long long)T * W * C);
  const AxisPlan pw = plan_axis((long long)B * H * T, W, C);
  if (int rc = run_axis<1 | 8 | 16>(gout, t1, pw, tp, wdev, nullptr, nullptr, bw, st)) return rc;
  if (int rc = run_axis<1 | 16>(t1, t2, pt, tp, wdev, nullptr, nullptr, none, st)) return rc;
  return run_axis<1 | 16>(t2, gx, ph, tp, wdev, nullptr, nullptr, none, st);
}

int smooth_fwd_bf16(int mode, const uint16_t* x, int B, int H, int T, int W, int C, const Taps& tp, const float* wdev,
                    uint16_t* out, float* maxval, uint32_t* ties, void* ws, cudaStream_t st) {
  KCCOT_CUDA(cudaMemsetAsync(ties, 0, kccot_smooth_ties_bytes(B, H, T, W, C), st));
  init_max_kernel<<<1, 1, 0, st>>>(maxval);
  KCCOT_LAUNCH_CHECK();
  const AxisPlan pt = plan_axis((long long)B * H, T, (long long)W * C);
  const Ties tie{ties, nullptr, nullptr};
  if (mode == 1) {
    if (int rc = run_axis_bf16<uint16_t, uint16_t, 2>(x, nullptr, pt, tp, wdev, maxval, nullptr, tie, st)) return rc;
    return run_axis_bf16<uint16_t, uint16_t, 1 | 4>(x, out, pt, tp, wdev, nullptr, maxval, tie, st);
  }
  // mode 3: bf16 -> fp32 H pass, the fp32 T pass and W max pass, fp32 -> bf16 W pass
  const size_t n = align_up((size_t)B * H * T * W * C * sizeof(float), 256);
  float* t1 = (float*)((char*)ws + 256);
  float* t2 = (float*)((char*)ws + 256 + n);
  const AxisPlan ph = plan_axis(B, H, (long long)T * W * C);
  const AxisPlan pw = plan_axis((long long)B * H * T, W, C);
  BwdIn none{};
  if (int rc = run_axis_bf16<uint16_t, float, 1>(x, t1, ph, tp, wdev, nullptr, nullptr, tie, st)) return rc;
  if (int rc = run_axis<1>(t1, t2, pt, tp, wdev, nullptr, nullptr, none, st)) return rc;
  if (int rc = run_axis<2>(t2, nullptr, pw, tp, wdev, maxval, nullptr, none, st)) return rc;
  return run_axis_bf16<float, uint16_t, 1 | 4>(t2, out, pw, tp, wdev, nullptr, maxval, tie, st);
}

int smooth_bwd_bf16(int mode, const uint16_t* gout, const uint16_t* out, const float* maxval, const uint32_t* ties,
                    int B, int H, int T, int W, int C, const Taps& tp, const float* wdev, uint16_t* gx, void* ws,
                    cudaStream_t st) {
  const long long nel = (long long)B * H * T * W * C;
  const long long nwords = (nel + 31) / 32;
  float* sums = (float*)ws;
  KCCOT_CUDA(cudaMemsetAsync(sums, 0, 2 * sizeof(float), st));
  tie_sums_bf16_kernel<<<(unsigned)min((long long)4 * num_sms(), (nel / 8 + FT - 1) / FT + 1), FT, 0, st>>>(
      gout, out, ties, nel, nwords, sums);
  KCCOT_LAUNCH_CHECK();
  const Ties tie{const_cast<uint32_t*>(ties), maxval, sums};     // read only: MODE & 4 is not set in the backward
  const AxisPlan pt = plan_axis((long long)B * H, T, (long long)W * C);
  if (mode == 1) return run_axis_bf16<uint16_t, uint16_t, 1 | 8 | 16>(gout, gx, pt, tp, wdev, nullptr, nullptr, tie, st);
  // mode 3: bf16 -> fp32 W pass with the tie transform, the fp32 T pass, fp32 -> bf16 H pass
  const size_t n = align_up((size_t)nel * sizeof(float), 256);
  float* t1 = (float*)((char*)ws + 256);
  float* t2 = (float*)((char*)ws + 256 + n);
  const AxisPlan ph = plan_axis(B, H, (long long)T * W * C);
  const AxisPlan pw = plan_axis((long long)B * H * T, W, C);
  BwdIn none{};
  if (int rc = run_axis_bf16<uint16_t, float, 1 | 8 | 16>(gout, t1, pw, tp, wdev, nullptr, nullptr, tie, st)) return rc;
  if (int rc = run_axis<1 | 16>(t1, t2, pt, tp, wdev, nullptr, nullptr, none, st)) return rc;
  return run_axis_bf16<float, uint16_t, 1 | 16>(t2, gx, ph, tp, wdev, nullptr, nullptr, tie, st);
}

// ---- batched independent problems -----------------------------------------------------------------------------------
// nprob videos [B,H,T,W,C], contiguous as [nprob, B,H,T,W,C], each filtered with its own 2R+1 device weights (row p of
// taps) and divided by its own maximum (maxval[p]).  The problem is blockIdx.y, so a CTA never spans two problems: its
// weights, its max atomic, its divisor and its tie sums are those of one problem, with no segmented reduction.  Every
// pass is planned per problem with plan_axis and, per element, forms its sums with the coefficients and the FMA order of
// the single-problem kernels, so problem p's numbers are those of a single-problem call on it.  One template serves
// fp32 and bf16 through TI / TO, as axis_col_bf16_kernel does; they are kernels of their own so that the single-problem
// kernels keep their code.  The backward's tie set is out == 1.0f where its first pass reads fp32 (TI = float) and the
// tie mask where it reads bf16; bit p * n + e of the mask is element e of problem p (the bf16 forward's last pass sets
// it, TO = uint16_t).
struct Batch {
  long long n;            // elements per problem
  const float* taps;      // [nprob][2R+1]
  float* maxval;          // [nprob]: reduced by MODE & 2, the divisor of MODE & 4, the m of MODE & 8
  const float* sums;      // [nprob][2]: sum(gout*out), number of tied maxima (MODE & 8)
  const float* out;       // fp32 forward output: the tie set of MODE & 8 with TI = float
  uint32_t* bits;         // the bf16 tie mask over all problems
};

template <int R>
__device__ __forceinline__ void load_batch_weights(float (&w)[2 * R + 1], const float* taps, int prob) {
#pragma unroll
  for (int k = 0; k < 2 * R + 1; ++k) w[k] = taps[prob * (2 * R + 1) + k];
}
// the BwdIn transform of the fp32 kernels on VecF
template <int V>
__device__ __forceinline__ void bwd_out_v(VecF<V>& r, float sc, float tie, const float* o) {
  VecF<V> t;
  load_v<V>(t, o);
#pragma unroll
  for (int j = 0; j < V; ++j) r.v[j] = r.v[j] * sc + ((t.v[j] == 1.0f) ? tie : 0.f);
}
// the input transform of a pass: the tie gradient on the first adjoint pass (MODE & 8); e: element index in the batch
template <typename TI, int MODE, int V>
__device__ __forceinline__ void batch_in(VecF<V>& r, float sc, float tie, const Batch& bt, long long e) {
  if constexpr ((MODE & 8) != 0) {
    if constexpr (sizeof(TI) == 4) bwd_out_v<V>(r, sc, tie, bt.out + e);
    else bwd_v<V>(r, sc, tie, bt.bits, e);
  }
}

template <typename TI, typename TO, int MODE, int V, int R>
__global__ void __launch_bounds__(FT) axis_col_batched_kernel(const TI* __restrict__ in, TO* __restrict__ out,
                                                              long long outer, int n, long long inner, Batch bt) {
  constexpr int kR = R, kTaps = 2 * R + 1;
  extern __shared__ float coef[];                          // coef[p][d] = A[p][p + d - R] (0 outside the matrix)
  const int prob = blockIdx.y;
  const long long off = (long long)prob * bt.n;
  float w[kTaps];
  load_batch_weights<R>(w, bt.taps, prob);
  for (int e = threadIdx.x; e < n * kTaps; e += FT) {
    const int p = e / kTaps, q = p + (e % kTaps) - kR;
    coef[e] = (q >= 0 && q < n) ? band_coef<R>(w, n, p, q, (MODE & 16) != 0) : 0.f;
  }
  __syncthreads();
  const long long iv = inner / V;
  const long long gid = (long long)blockIdx.x * FT + threadIdx.x;
  float lmax = -3.0e38f;
  if (gid < outer * iv) {
    const long long o = gid / iv;
    const long long base = off + o * n * inner + (gid - o * iv) * V;
    float gscale = 0.f, gtie = 0.f, inv = 1.f;
    if (MODE & 8) {
      const float m = bt.maxval[prob];
      gscale = 1.f / m;
      gtie = -(bt.sums[2 * prob] / m) / bt.sums[2 * prob + 1];
    }
    if (MODE & 4) inv = bt.maxval[prob];
    auto fetch = [&](int q) {
      VecF<V> r;
      if (q < n) {
        load_v<V>(r, in + base + (long long)q * inner);
        batch_in<TI, MODE, V>(r, gscale, gtie, bt, base + (long long)q * inner);
      } else {
#pragma unroll
        for (int j = 0; j < V; ++j) r.v[j] = 0.f;
      }
      return r;
    };
    VecF<V> win[kTaps];
#pragma unroll
    for (int d = 0; d < kR; ++d)
#pragma unroll
      for (int j = 0; j < V; ++j) win[d].v[j] = 0.f;
#pragma unroll
    for (int d = kR; d < kTaps; ++d) win[d] = fetch(d - kR);
    constexpr bool kDeep = V * kTaps <= 64;
    VecF<V> next = fetch(kR + 1), next2;
    for (int p = 0; p < n; ++p) {
      if constexpr (kDeep) next2 = fetch(p + kR + 2);
      VecF<V> acc;
#pragma unroll
      for (int j = 0; j < V; ++j) acc.v[j] = 0.f;
#pragma unroll
      for (int d = 0; d < kTaps; ++d) {
        const float c = coef[p * kTaps + d];
#pragma unroll
        for (int j = 0; j < V; ++j) acc.v[j] = fmaf(c, win[d].v[j], acc.v[j]);
      }
      if (MODE & 4) {
#pragma unroll
        for (int j = 0; j < V; ++j) acc.v[j] /= inv;
        if constexpr (sizeof(TO) == 2) mark_ties<V>(bt.bits, acc, base + (long long)p * inner);
      }
      if (MODE & 2) {
#pragma unroll
        for (int j = 0; j < V; ++j) lmax = fmaxf(lmax, acc.v[j]);
      }
      if (MODE & 1) store_v<V>(out + base + (long long)p * inner, acc);
#pragma unroll
      for (int d = 0; d < kTaps - 1; ++d) win[d] = win[d + 1];
      win[kTaps - 1] = next;
      if constexpr (kDeep) next = next2;
      else next = fetch(p + kR + 2);
    }
  }
  if (MODE & 2) {
    lmax = warp_max(lmax);
    if ((threadIdx.x & 31) == 0) atomic_max_float(bt.maxval + prob, lmax);
  }
}

template <typename TI, typename TO, int MODE, int R>
__global__ void __launch_bounds__(1024) axis_tile_batched_kernel(const TI* __restrict__ in, TO* __restrict__ out,
                                                                 long long outer, int n, int inner, int o_chunk,
                                                                 Batch bt) {
  constexpr int kR = R, kTaps = 2 * R + 1;
  extern __shared__ __align__(16) float tile[];            // [o_chunk][n][inner], contiguous like global memory
  const int prob = blockIdx.y;
  const int ni = n * inner;
  const long long o0 = (long long)blockIdx.x * o_chunk;
  const int no = (int)min((long long)o_chunk, outer - o0);
  const long long g0 = (long long)prob * bt.n + o0 * ni;    // element index in the batch
  const int telems = no * ni;
  float gscale = 0.f, gtie = 0.f, inv = 1.f;
  if (MODE & 8) {
    const float m = bt.maxval[prob];
    gscale = 1.f / m;
    gtie = -(bt.sums[2 * prob] / m) / bt.sums[2 * prob + 1];
  }
  if (MODE & 4) inv = bt.maxval[prob];
  // the widest loads the tile's row length and the pointers allow (g0 % 8 == 0 whenever ni % 8 == 0)
  auto fill = [&](auto vw) {
    constexpr int VV = decltype(vw)::value;
    for (int e = threadIdx.x * VV; e < telems; e += blockDim.x * VV) {
      VecF<VV> r;
      load_v<VV>(r, in + g0 + e);
      batch_in<TI, MODE, VV>(r, gscale, gtie, bt, g0 + e);
      store_v<VV>(tile + e, r);
    }
  };
  auto aligned = [&](int v) {
    const uintptr_t a = (uintptr_t)(v * sizeof(TI) < 16 ? v * sizeof(TI) : 16) - 1;
    return ni % v == 0 && (reinterpret_cast<uintptr_t>(in + g0) & a) == 0 &&
           (!(MODE & 8) || sizeof(TI) == 2 || (reinterpret_cast<uintptr_t>(bt.out + g0) & (v == 1 ? 3 : 15)) == 0);
  };
  if (aligned(8)) fill(std::integral_constant<int, 8>());
  else if (aligned(4)) fill(std::integral_constant<int, 4>());
  else fill(std::integral_constant<int, 1>());
  const int t = threadIdx.x;
  float c[kTaps];
  int off[kTaps];
  {
    const int p = min(t, ni - 1) / inner;
    float w[kTaps];
    load_batch_weights<R>(w, bt.taps, prob);
#pragma unroll
    for (int d = 0; d < kTaps; ++d) {
      const int q = p + d - kR;
      const bool ok = q >= 0 && q < n;
      c[d] = ok ? band_coef<R>(w, n, p, q, (MODE & 16) != 0) : 0.f;
      off[d] = ok ? (d - kR) * inner : 0;
    }
  }
  __syncthreads();
  float lmax = -3.0e38f;
  auto row_out = [&](int oo) {
    const float* row = tile + oo * ni + t;
    VecF<1> acc;
    acc.v[0] = 0.f;
#pragma unroll
    for (int d = 0; d < kTaps; ++d) acc.v[0] = fmaf(c[d], row[off[d]], acc.v[0]);
    const long long e = g0 + (long long)oo * ni + t;
    if (MODE & 4) {
      acc.v[0] = acc.v[0] / inv;
      if constexpr (sizeof(TO) == 2) mark_ties<1>(bt.bits, acc, e);
    }
    if (MODE & 2) lmax = fmaxf(lmax, acc.v[0]);
    if (MODE & 1) store_v<1>(out + e, acc);
  };
  if (t < ni) {
    if constexpr ((MODE & 2) != 0) {
#pragma unroll 1
      for (int oo = 0; oo < no; ++oo) row_out(oo);
    } else {
      for (int oo = 0; oo < no; ++oo) row_out(oo);
    }
  }
  if (MODE & 2) {
    lmax = warp_max(lmax);
    if ((threadIdx.x & 31) == 0) atomic_max_float(bt.maxval + prob, lmax);
  }
}

__global__ void init_max_batched_kernel(float* m, int nprob) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nprob) m[i] = __int_as_float(0xff800000);
}

// sums[2p] = sum gout * out over problem p (blockIdx.y), sums[2p+1] = its number of tied maxima: out == 1.0f in fp32,
// the popcount of the mask bits p*n .. p*n + n - 1 in bf16 (a word may hold bits of two problems)
template <typename T>
__global__ void __launch_bounds__(FT) tie_sums_batched_kernel(const T* __restrict__ gout, const T* __restrict__ out,
                                                              const uint32_t* __restrict__ bits, long long n,
                                                              float* sums) {
  constexpr int V = 16 / sizeof(T);                        // elements per 16-byte access
  const int prob = blockIdx.y;
  const long long off = (long long)prob * n;
  gout += off;
  out += off;
  float s = 0.f, c = 0.f;
  const long long stride = (long long)gridDim.x * FT;
  const long long tid = (long long)blockIdx.x * FT + threadIdx.x;
  const bool vec = ((reinterpret_cast<uintptr_t>(gout) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  const long long nv = vec ? n / V : 0;
  auto acc = [&](const VecF<V>& g, const VecF<V>& o) {
#pragma unroll
    for (int j = 0; j < V; ++j) s = fmaf(g.v[j], o.v[j], s);
    if constexpr (sizeof(T) == 4) {
#pragma unroll
      for (int j = 0; j < V; ++j) c += (o.v[j] == 1.0f ? 1.f : 0.f);
    }
  };
  long long i = tid;
  for (; i + 3 * stride < nv; i += 4 * stride) {
    VecF<V> g[4], o[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { load_v<V>(g[u], gout + (i + u * stride) * V); load_v<V>(o[u], out + (i + u * stride) * V); }
#pragma unroll
    for (int u = 0; u < 4; ++u) acc(g[u], o[u]);
  }
  for (; i < nv; i += stride) {
    VecF<V> g, o;
    load_v<V>(g, gout + i * V);
    load_v<V>(o, out + i * V);
    acc(g, o);
  }
  for (long long k = V * nv + tid; k < n; k += stride) {
    VecF<1> g, o;
    load_v<1>(g, gout + k);
    load_v<1>(o, out + k);
    s = fmaf(g.v[0], o.v[0], s);
    if constexpr (sizeof(T) == 4) c += (o.v[0] == 1.0f) ? 1.f : 0.f;
  }
  if constexpr (sizeof(T) == 2) {
    const long long lo = off, hi = off + n, w0 = lo >> 5, w1 = (hi - 1) >> 5;
    unsigned cnt = 0;
    for (long long w = w0 + tid; w <= w1; w += stride) {
      uint32_t b = bits[w];
      if (w == w0) b &= ~0u << (lo & 31);
      if (w == w1 && (hi & 31)) b &= (1u << (hi & 31)) - 1u;
      cnt += __popc(b);
    }
    c = (float)cnt;
  }
  __shared__ float red[2][FT / 32];
  s = warp_sum(s);
  c = warp_sum(c);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s; red[1][threadIdx.x >> 5] = c; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float ss = 0.f, cc = 0.f;
#pragma unroll
    for (int w = 0; w < FT / 32; ++w) { ss += red[0][w]; cc += red[1][w]; }
    atomicAdd(&sums[2 * prob], ss);
    atomicAdd(&sums[2 * prob + 1], cc);
  }
}

// one pass over all problems; p is the plan of one problem, which a single-problem call of that shape would use (its
// tile / column choice and vector width)
template <typename TI, typename TO, int MODE, int R>
int run_batched_r(const TI* in, TO* out, const AxisPlan& p, int nprob, const Batch& bt, cudaStream_t st) {
  if (p.tiled) {
    const int ni = p.n * (int)p.inner;
    const int threads = (ni + 31) / 32 * 32;
    const dim3 grid((unsigned)((p.outer + p.o_chunk - 1) / p.o_chunk), (unsigned)nprob);
    const size_t smem = (size_t)p.o_chunk * ni * sizeof(float);
    axis_tile_batched_kernel<TI, TO, MODE, R><<<grid, threads, smem, st>>>(in, out, p.outer, p.n, (int)p.inner,
                                                                          p.o_chunk, bt);
  } else {
    // n % v == 0 when inner % v == 0, so every problem's rows have the alignment of problem 0's
    auto fits = [&](int v) {
      const uintptr_t a = (uintptr_t)(v * sizeof(TI) < 16 ? v * sizeof(TI) : 16) - 1;
      const uintptr_t b = (uintptr_t)(v * sizeof(TO) < 16 ? v * sizeof(TO) : 16) - 1;
      return p.inner % v == 0 && (reinterpret_cast<uintptr_t>(in) & a) == 0 &&
             (!(MODE & 1) || (reinterpret_cast<uintptr_t>(out) & b) == 0) &&
             (!(MODE & 8) || sizeof(TI) == 2 || (reinterpret_cast<uintptr_t>(bt.out) & a) == 0);
    };
    constexpr bool kF32 = sizeof(TI) == 4 && sizeof(TO) == 4;      // the fp32 kernels' widths: 4 or 1
    const int v = kF32 ? (fits(4) ? 4 : 1)
                       : fits(8) && p.outer * (p.inner / 8) >= 1024LL * num_sms() ? 8 : fits(4) ? 4 : fits(8) ? 8 : 1;
    const long long total = p.outer * (p.inner / v);
    const dim3 grid((unsigned)((total + FT - 1) / FT), (unsigned)nprob);
    const size_t smem = (size_t)p.n * (2 * R + 1) * sizeof(float);
    void (*kernel)(const TI*, TO*, long long, int, long long, Batch) =
        v == 4 ? axis_col_batched_kernel<TI, TO, MODE, 4, R> : axis_col_batched_kernel<TI, TO, MODE, 1, R>;
    if constexpr (!kF32) {
      if (v == 8) kernel = axis_col_batched_kernel<TI, TO, MODE, 8, R>;
    }
    if (smem > 48 * 1024)
      KCCOT_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<grid, FT, smem, st>>>(in, out, p.outer, p.n, p.inner, bt);
  }
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}
template <typename TI, typename TO, int MODE>
int run_batched(const TI* in, TO* out, const AxisPlan& p, int nprob, int radius, const Batch& bt, cudaStream_t st) {
  switch (radius) {
    case 1: return run_batched_r<TI, TO, MODE, 1>(in, out, p, nprob, bt, st);
    case 2: return run_batched_r<TI, TO, MODE, 2>(in, out, p, nprob, bt, st);
    case 3: return run_batched_r<TI, TO, MODE, 3>(in, out, p, nprob, bt, st);
    case 4: return run_batched_r<TI, TO, MODE, 4>(in, out, p, nprob, bt, st);
    case 5: return run_batched_r<TI, TO, MODE, 5>(in, out, p, nprob, bt, st);
    case 6: return run_batched_r<TI, TO, MODE, 6>(in, out, p, nprob, bt, st);
  }
  set_error("smoothing radius %d not supported (1..%d)", radius, kMaxRadius);
  return KCCOT_EUNSUPPORTED;
}

constexpr int kMaxProblems = 65535;                           // gridDim.y
size_t batched_head_bytes(int nprob) { return align_up((size_t)nprob * 2 * sizeof(float), 256); }

// argument checks of the batched entries: those of the *_dev entries plus the problem count and the batched workspace
int smooth_batched_args(int mode, int nprob, int B, int H, int T, int W, int C, const float* taps, int radius,
                        bool need_ws, void* ws, size_t ws_bytes, Taps* tp) {
  KCCOT_CHECK_ARG(nprob >= 1 && nprob <= kMaxProblems, "nprob must be in 1..%d (nprob=%d)", kMaxProblems, nprob);
  if (int rc = smooth_args(mode, B, H, T, W, C, taps, radius, taps, radius, true, ws, ws_bytes, tp)) return rc;
  if (need_ws)
    KCCOT_CHECK_ARG(ws && ws_bytes >= kccot_smooth_batched_workspace_bytes(mode, nprob, B, H, T, W, C),
                    "workspace too small");
  KCCOT_CHECK_ARG((reinterpret_cast<uintptr_t>(ws) & 15) == 0, "workspace must be 16-byte aligned");
  return KCCOT_OK;
}

// T = float (fp32 videos) or uint16_t (bf16); ties is used by bf16 only
template <typename T>
int smooth_batched_fwd(int mode, const T* x, int nprob, int B, int H, int T_, int W, int C, const float* taps,
                       int radius, T* out, float* maxval, uint32_t* ties, void* ws, cudaStream_t st) {
  const long long n = (long long)B * H * T_ * W * C;
  constexpr bool kBf16 = sizeof(T) == 2;
  if (kBf16) KCCOT_CUDA(cudaMemsetAsync(ties, 0, ((size_t)nprob * n + 31) / 32 * sizeof(uint32_t), st));
  init_max_batched_kernel<<<(nprob + 255) / 256, 256, 0, st>>>(maxval, nprob);
  KCCOT_LAUNCH_CHECK();
  const Batch bt{n, taps, maxval, nullptr, nullptr, ties};
  const AxisPlan pt = plan_axis((long long)B * H, T_, (long long)W * C);
  if (mode == 1) {
    if (int rc = run_batched<T, T, 2>(x, nullptr, pt, nprob, radius, bt, st)) return rc;
    return run_batched<T, T, 1 | 4>(x, out, pt, nprob, radius, bt, st);
  }
  const size_t head = batched_head_bytes(nprob), sz = align_up((size_t)nprob * n * sizeof(float), 256);
  float* t1 = (float*)((char*)ws + head);
  float* t2 = (float*)((char*)ws + head + sz);
  const AxisPlan ph = plan_axis(B, H, (long long)T_ * W * C);
  const AxisPlan pw = plan_axis((long long)B * H * T_, W, C);
  if (int rc = run_batched<T, float, 1>(x, t1, ph, nprob, radius, bt, st)) return rc;
  if (int rc = run_batched<float, float, 1>(t1, t2, pt, nprob, radius, bt, st)) return rc;
  if (int rc = run_batched<float, float, 2>(t2, nullptr, pw, nprob, radius, bt, st)) return rc;
  return run_batched<float, T, 1 | 4>(t2, out, pw, nprob, radius, bt, st);
}

template <typename T>
int smooth_batched_bwd(int mode, const T* gout, const T* out, const float* maxval, const uint32_t* ties, int nprob,
                       int B, int H, int T_, int W, int C, const float* taps, int radius, T* gx, void* ws,
                       cudaStream_t st) {
  const long long n = (long long)B * H * T_ * W * C;
  float* sums = (float*)ws;
  KCCOT_CUDA(cudaMemsetAsync(sums, 0, (size_t)nprob * 2 * sizeof(float), st));
  {
    const long long single = min((long long)4 * num_sms(), (n / (16 / (long long)sizeof(T)) + FT - 1) / FT + 1);
    const long long per = max(1LL, min(single, (8LL * num_sms() + nprob - 1) / nprob));
    tie_sums_batched_kernel<T><<<dim3((unsigned)per, (unsigned)nprob), FT, 0, st>>>(gout, out, ties, n, sums);
    KCCOT_LAUNCH_CHECK();
  }
  // read only: no pass of the backward sets MODE & 4
  const Batch bt{n, taps, const_cast<float*>(maxval), sums, sizeof(T) == 4 ? (const float*)out : nullptr,
                 const_cast<uint32_t*>(ties)};
  const AxisPlan pt = plan_axis((long long)B * H, T_, (long long)W * C);
  if (mode == 1) return run_batched<T, T, 1 | 8 | 16>(gout, gx, pt, nprob, radius, bt, st);
  const size_t head = batched_head_bytes(nprob), sz = align_up((size_t)nprob * n * sizeof(float), 256);
  float* t1 = (float*)((char*)ws + head);
  float* t2 = (float*)((char*)ws + head + sz);
  const AxisPlan ph = plan_axis(B, H, (long long)T_ * W * C);
  const AxisPlan pw = plan_axis((long long)B * H * T_, W, C);
  if (int rc = run_batched<T, float, 1 | 8 | 16>(gout, t1, pw, nprob, radius, bt, st)) return rc;
  if (int rc = run_batched<float, float, 1 | 16>(t1, t2, pt, nprob, radius, bt, st)) return rc;
  return run_batched<float, T, 1 | 16>(t2, gx, ph, nprob, radius, bt, st);
}
}  // namespace
}  // namespace kccot

using namespace kccot;

extern "C" {

size_t kccot_smooth_workspace_bytes(int mode, int B, int H, int T, int W, int C) {
  const size_t n = (size_t)B * H * T * W * C * sizeof(float);
  return align_up(256 + (mode == 3 ? 2 * align_up(n, 256) : 0), 256);
}

int kccot_smooth_fwd(int mode, const float* x, int B, int H, int T, int W, int C, const float* taps_t, int radius_t,
                     const float* taps_s, int radius_s, float* out, float* maxval, void* ws, size_t ws_bytes, void* stream) {
  KCCOT_CHECK_ARG(mode == 1 || mode == 3, "smoothing mode must be 1 (temporal) or 3 (3-D); the reference's '2d' "
                                          "branch raises (data_utils.py:537-538)");
  KCCOT_CHECK_ARG(x && out && maxval, "null pointer");
  KCCOT_CHECK_ARG(B >= 1 && H >= 1 && T >= 1 && W >= 1 && C >= 1, "bad sizes");
  KCCOT_CHECK_ARG(T <= kMaxAxis && H <= kMaxAxis && W <= kMaxAxis, "axis longer than %d not supported (H=%d T=%d W=%d)", kMaxAxis,
                  H, T, W);
  Taps tp;
  if (int rc = mode == 1 ? make_taps(&tp, taps_t, radius_t, "temporal_convolution") : make_taps(&tp, taps_s, radius_s,
                                                                                             "gaussian_convolution3D"))
    return rc;
  KCCOT_CHECK_ARG(T > tp.r, "REFLECT padding by %d needs T > %d (T=%d)", tp.r, tp.r, T);
  return smooth_fwd_f32(mode, x, B, H, T, W, C, tp, nullptr, out, maxval, ws, ws_bytes, (cudaStream_t)stream);
}

int kccot_smooth_bwd(int mode, const float* gout, const float* out, const float* maxval, int B, int H, int T, int W,
                     int C, const float* taps_t, int radius_t, const float* taps_s, int radius_s, float* gx, void* ws,
                     size_t ws_bytes, void* stream) {
  KCCOT_CHECK_ARG(mode == 1 || mode == 3, "smoothing mode must be 1 or 3");
  KCCOT_CHECK_ARG(gout && out && maxval && gx && ws && ws_bytes >= 256, "null pointer / workspace");
  Taps tp;
  if (int rc = mode == 1 ? make_taps(&tp, taps_t, radius_t, "temporal_convolution") : make_taps(&tp, taps_s, radius_s,
                                                                                             "gaussian_convolution3D"))
    return rc;
  return smooth_bwd_f32(mode, gout, out, maxval, B, H, T, W, C, tp, nullptr, gx, ws, ws_bytes, (cudaStream_t)stream);
}

int kccot_smooth_fwd_dev(int mode, const float* x, int B, int H, int T, int W, int C, const float* taps_dev, int radius,
                         float* out, float* maxval, void* ws, size_t ws_bytes, void* stream) {
  KCCOT_CHECK_ARG(mode == 1 || mode == 3, "smoothing mode must be 1 (temporal) or 3 (3-D); the reference's '2d' "
                                          "branch raises (data_utils.py:537-538)");
  KCCOT_CHECK_ARG(x && out && maxval, "null pointer");
  Taps tp;
  if (int rc = smooth_args(mode, B, H, T, W, C, taps_dev, radius, taps_dev, radius, true, ws, ws_bytes, &tp)) return rc;
  return smooth_fwd_f32(mode, x, B, H, T, W, C, tp, taps_dev, out, maxval, ws, ws_bytes, (cudaStream_t)stream);
}

int kccot_smooth_bwd_dev(int mode, const float* gout, const float* out, const float* maxval, int B, int H, int T, int W,
                         int C, const float* taps_dev, int radius, float* gx, void* ws, size_t ws_bytes, void* stream) {
  KCCOT_CHECK_ARG(mode == 1 || mode == 3, "smoothing mode must be 1 or 3");
  KCCOT_CHECK_ARG(gout && out && maxval && gx && ws && ws_bytes >= 256, "null pointer / workspace");
  Taps tp;
  if (int rc = smooth_args(mode, B, H, T, W, C, taps_dev, radius, taps_dev, radius, true, ws, ws_bytes, &tp)) return rc;
  return smooth_bwd_f32(mode, gout, out, maxval, B, H, T, W, C, tp, taps_dev, gx, ws, ws_bytes, (cudaStream_t)stream);
}

size_t kccot_smooth_ties_bytes(int B, int H, int T, int W, int C) {
  if (B < 1 || H < 1 || T < 1 || W < 1 || C < 1) return 0;
  const size_t n = (size_t)B * H * T * W * C;
  return (n + 31) / 32 * sizeof(uint32_t);
}

int kccot_smooth_fwd_bf16(int mode, const uint16_t* x, int B, int H, int T, int W, int C, const float* taps_t,
                          int radius_t, const float* taps_s, int radius_s, uint16_t* out, float* maxval,
                          uint32_t* ties, void* ws, size_t ws_bytes, void* stream) {
  KCCOT_CHECK_ARG(mode == 1 || mode == 3, "smoothing mode must be 1 (temporal) or 3 (3-D); the reference's '2d' "
                                          "branch raises (data_utils.py:537-538)");
  KCCOT_CHECK_ARG(x && out && maxval && ties, "null pointer");
  KCCOT_CHECK_ARG((reinterpret_cast<uintptr_t>(ties) & 3) == 0, "tie mask must be 4-byte aligned");
  Taps tp;
  if (int rc = smooth_args(mode, B, H, T, W, C, taps_t, radius_t, taps_s, radius_s, false, ws, ws_bytes, &tp)) return rc;
  return smooth_fwd_bf16(mode, x, B, H, T, W, C, tp, nullptr, out, maxval, ties, ws, (cudaStream_t)stream);
}

int kccot_smooth_bwd_bf16(int mode, const uint16_t* gout, const uint16_t* out, const float* maxval,
                          const uint32_t* ties, int B, int H, int T, int W, int C, const float* taps_t, int radius_t,
                          const float* taps_s, int radius_s, uint16_t* gx, void* ws, size_t ws_bytes, void* stream) {
  KCCOT_CHECK_ARG(mode == 1 || mode == 3, "smoothing mode must be 1 or 3");
  KCCOT_CHECK_ARG(gout && out && maxval && ties && gx && ws && ws_bytes >= 256, "null pointer / workspace");
  KCCOT_CHECK_ARG((reinterpret_cast<uintptr_t>(ties) & 3) == 0, "tie mask must be 4-byte aligned");
  Taps tp;
  if (int rc = smooth_args(mode, B, H, T, W, C, taps_t, radius_t, taps_s, radius_s, false, ws, ws_bytes, &tp)) return rc;
  return smooth_bwd_bf16(mode, gout, out, maxval, ties, B, H, T, W, C, tp, nullptr, gx, ws, (cudaStream_t)stream);
}

int kccot_smooth_fwd_bf16_dev(int mode, const uint16_t* x, int B, int H, int T, int W, int C, const float* taps_dev,
                              int radius, uint16_t* out, float* maxval, uint32_t* ties, void* ws, size_t ws_bytes,
                              void* stream) {
  KCCOT_CHECK_ARG(mode == 1 || mode == 3, "smoothing mode must be 1 (temporal) or 3 (3-D); the reference's '2d' "
                                          "branch raises (data_utils.py:537-538)");
  KCCOT_CHECK_ARG(x && out && maxval && ties, "null pointer");
  KCCOT_CHECK_ARG((reinterpret_cast<uintptr_t>(ties) & 3) == 0, "tie mask must be 4-byte aligned");
  Taps tp;
  if (int rc = smooth_args(mode, B, H, T, W, C, taps_dev, radius, taps_dev, radius, true, ws, ws_bytes, &tp)) return rc;
  return smooth_fwd_bf16(mode, x, B, H, T, W, C, tp, taps_dev, out, maxval, ties, ws, (cudaStream_t)stream);
}

int kccot_smooth_bwd_bf16_dev(int mode, const uint16_t* gout, const uint16_t* out, const float* maxval,
                              const uint32_t* ties, int B, int H, int T, int W, int C, const float* taps_dev, int radius,
                              uint16_t* gx, void* ws, size_t ws_bytes, void* stream) {
  KCCOT_CHECK_ARG(mode == 1 || mode == 3, "smoothing mode must be 1 or 3");
  KCCOT_CHECK_ARG(gout && out && maxval && ties && gx && ws && ws_bytes >= 256, "null pointer / workspace");
  KCCOT_CHECK_ARG((reinterpret_cast<uintptr_t>(ties) & 3) == 0, "tie mask must be 4-byte aligned");
  Taps tp;
  if (int rc = smooth_args(mode, B, H, T, W, C, taps_dev, radius, taps_dev, radius, true, ws, ws_bytes, &tp)) return rc;
  return smooth_bwd_bf16(mode, gout, out, maxval, ties, B, H, T, W, C, tp, taps_dev, gx, ws, (cudaStream_t)stream);
}

size_t kccot_smooth_batched_workspace_bytes(int mode, int nprob, int B, int H, int T, int W, int C) {
  if (nprob < 1 || B < 1 || H < 1 || T < 1 || W < 1 || C < 1) return 0;
  const size_t n = (size_t)nprob * B * H * T * W * C * sizeof(float);
  return batched_head_bytes(nprob) + (mode == 3 ? 2 * align_up(n, 256) : 0);
}

int kccot_smooth_batched_fwd(int mode, const float* x, int nprob, int B, int H, int T, int W, int C,
                             const float* taps_dev, int radius, float* out, float* maxval, void* ws, size_t ws_bytes,
                             void* stream) {
  KCCOT_CHECK_ARG(mode == 1 || mode == 3, "smoothing mode must be 1 (temporal) or 3 (3-D); the reference's '2d' "
                                          "branch raises (data_utils.py:537-538)");
  KCCOT_CHECK_ARG(x && out && maxval, "null pointer");
  Taps tp;
  if (int rc = smooth_batched_args(mode, nprob, B, H, T, W, C, taps_dev, radius, mode == 3, ws, ws_bytes, &tp))
    return rc;
  return smooth_batched_fwd<float>(mode, x, nprob, B, H, T, W, C, taps_dev, radius, out, maxval, nullptr, ws,
                                   (cudaStream_t)stream);
}

int kccot_smooth_batched_bwd(int mode, const float* gout, const float* out, const float* maxval, int nprob, int B,
                             int H, int T, int W, int C, const float* taps_dev, int radius, float* gx, void* ws,
                             size_t ws_bytes, void* stream) {
  KCCOT_CHECK_ARG(mode == 1 || mode == 3, "smoothing mode must be 1 or 3");
  KCCOT_CHECK_ARG(gout && out && maxval && gx && ws, "null pointer / workspace");
  Taps tp;
  if (int rc = smooth_batched_args(mode, nprob, B, H, T, W, C, taps_dev, radius, true, ws, ws_bytes, &tp)) return rc;
  return smooth_batched_bwd<float>(mode, gout, out, maxval, nullptr, nprob, B, H, T, W, C, taps_dev, radius, gx, ws,
                                   (cudaStream_t)stream);
}

int kccot_smooth_batched_fwd_bf16(int mode, const uint16_t* x, int nprob, int B, int H, int T, int W, int C,
                                  const float* taps_dev, int radius, uint16_t* out, float* maxval, uint32_t* ties,
                                  void* ws, size_t ws_bytes, void* stream) {
  KCCOT_CHECK_ARG(mode == 1 || mode == 3, "smoothing mode must be 1 (temporal) or 3 (3-D); the reference's '2d' "
                                          "branch raises (data_utils.py:537-538)");
  KCCOT_CHECK_ARG(x && out && maxval && ties, "null pointer");
  KCCOT_CHECK_ARG((reinterpret_cast<uintptr_t>(ties) & 3) == 0, "tie mask must be 4-byte aligned");
  Taps tp;
  if (int rc = smooth_batched_args(mode, nprob, B, H, T, W, C, taps_dev, radius, mode == 3, ws, ws_bytes, &tp))
    return rc;
  return smooth_batched_fwd<uint16_t>(mode, x, nprob, B, H, T, W, C, taps_dev, radius, out, maxval, ties, ws,
                                      (cudaStream_t)stream);
}

int kccot_smooth_batched_bwd_bf16(int mode, const uint16_t* gout, const uint16_t* out, const float* maxval,
                                  const uint32_t* ties, int nprob, int B, int H, int T, int W, int C,
                                  const float* taps_dev, int radius, uint16_t* gx, void* ws, size_t ws_bytes,
                                  void* stream) {
  KCCOT_CHECK_ARG(mode == 1 || mode == 3, "smoothing mode must be 1 or 3");
  KCCOT_CHECK_ARG(gout && out && maxval && ties && gx && ws, "null pointer / workspace");
  KCCOT_CHECK_ARG((reinterpret_cast<uintptr_t>(ties) & 3) == 0, "tie mask must be 4-byte aligned");
  Taps tp;
  if (int rc = smooth_batched_args(mode, nprob, B, H, T, W, C, taps_dev, radius, true, ws, ws_bytes, &tp)) return rc;
  return smooth_batched_bwd<uint16_t>(mode, gout, out, maxval, ties, nprob, B, H, T, W, C, taps_dev, radius, gx, ws,
                                      (cudaStream_t)stream);
}

}  // extern "C"
