// Sinkhorn for B <= 64: one CTA per problem, everything on chip for all L iterations
// (gan_utils.py:151-164), and the fully unrolled reverse pass (SURVEY.md Appendix A) with the
// adjoint of C accumulated in registers.
//
// 4 threads share a row (or a column): thread (i, q) owns the row slice C[i][q*EPT .. q*EPT+EPT) and
// the column slice C[q*EPT .. q*EPT+EPT)[i], both in registers.  Internal units: log2 domain, cost
// shifted by its minimum:  Chat = (C - c0) * log2(e)/eps,  uhat = (u - c0) * log2(e)/eps,
// vhat = v * log2(e)/eps.
//
// FAST PATH (stabilised scaling form).  The log-domain update
//     uhat_i <- ahat - log2 sum_j exp2(vhat_j - Chat_ij)
// costs one ex2 per matrix element per half-iteration and is bound by the 16 MUFU lanes of an SM.
// With the kernel absorbed once at reference potentials,  Kt_ij = exp2(alpha_i - Chat_ij)
// (alpha_i = row minimum, so every row holds a 1), the same update is a mat-vec:
//     s_i = sum_j Kt_ij b_j,  b_j = exp2(vhat_j);   uhat_i = ahat + alpha_i - log2 s_i,
//     a_i = exp2(uhat_i - alpha_i) = 2^ahat / s_i;   t_j = sum_i Kt_ij a_i,  vhat_j = ahat - log2 t_j,
// i.e. ONE FMA per element and two MUFU ops per row.  The iterates are the same numbers (the
// algebra is exact); only rounding differs.  The backward pass uses the same trick with the kernel
// absorbed at the final potentials (Kt = pi): every softmax matrix of Appendix A is pi times a
// rank-one factor.
// SLOW PATH (guard).  If a scaling leaves [2^-90, 2^90] (ill-scaled cost / tiny eps) the forward rolls
// back one iteration and continues, for the rest of the solve, with the plain log-domain updates with
// max subtraction — the reference's formulation.  The backward switches to direct exponentials before
// any rank-one factor would leave 2^+-60.
#include <type_traits>

#include "common.cuh"
#include "sinkhorn.cuh"

namespace kccot {

namespace {
constexpr float kBig = 1e30f;      // padding cost: exp2(anything - kBig) == 0, and 0 * kBig == 0
constexpr float kLo = 8.0e-28f;    // ~2^-90
constexpr float kHi = 1.2e27f;     // ~2^90
constexpr float kExpLim = 60.f;    // |log2| allowed for a backward rank-one factor

// Lanes per row (and per column): a row of the B x B problem is split over LPR adjacent lanes, EPT elements
// each.  EPT = 8: four lanes (B <= 32); EPT = 16: four lanes (B <= 64, backward); EPT = 32: two lanes (B <= 64,
// forward) — one shuffle instead of two and a 4-warp barrier instead of an 8-warp one: 478 against 569 cycles
// per iteration of a bare mat-vec loop on a B200 (DESIGN.md §5).
__host__ __device__ constexpr int lpr_of(int ept) { return ept == 32 ? 2 : 4; }

template <int LPR>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = 1; o < LPR; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
template <int LPR>
__device__ __forceinline__ float group_max(float v) {
#pragma unroll
  for (int o = 1; o < LPR; o <<= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
template <int LPR>
__device__ __forceinline__ float group_min(float v) {
#pragma unroll
  for (int o = 1; o < LPR; o <<= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float fast_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ float block_reduce(float v, float* red, bool is_min) {
  v = is_min ? warp_min(v) : warp_sum(v);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float r = is_min ? kBig : 0.f;
  const int nw = (blockDim.x + 31) >> 5;
  for (int w = 0; w < nw; ++w) r = is_min ? fminf(r, red[w]) : r + red[w];
  return r;
}

// loads both register slices of C, shifted by its minimum and scaled to log2 units
template <int EPT>
__device__ __forceinline__ float load_slices(const float* __restrict__ Cn, int B, float kscale, float* red,
                                             float (&Cr)[EPT], float (&Cc)[EPT]) {
  constexpr int LPR = lpr_of(EPT);
  const int i = threadIdx.x / LPR, q = threadIdx.x % LPR;
  float mn = kBig;
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    const int j = q * EPT + e;
    Cr[e] = (i < B && j < B) ? Cn[(long long)i * B + j] : kBig;
    Cc[e] = (i < B && j < B) ? Cn[(long long)j * B + i] : kBig;
    mn = fminf(mn, Cr[e]);
  }
  const float c0 = block_reduce(mn, red, true);
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    Cr[e] = (Cr[e] < kBig) ? (Cr[e] - c0) * kscale : kBig;
    Cc[e] = (Cc[e] < kBig) ? (Cc[e] - c0) * kscale : kBig;
  }
  return c0;
}

// Same slices through a shared-memory tile: one batch of coalesced 16-byte loads of the whole matrix, then
// row and column slices out of shared memory (the direct version issues 2 x EPT scalar loads per thread, the
// column half of them strided by B: 3 700-3 900 cycles on the critical path of the forward kernel).
// `tile` needs B * (LPR*EPT + 4) floats and is free again when the function returns.
template <int EPT>
__device__ __forceinline__ float load_slices_tile(const float* __restrict__ Cn, int B, float kscale, float* red,
                                                  float (&Cr)[EPT], float (&Cc)[EPT], float* tile) {
  constexpr int LPR = lpr_of(EPT);
  constexpr int PS = LPR * EPT + 4;
  const int i = threadIdx.x / LPR, q = threadIdx.x % LPR;
  {
    const float4* C4 = reinterpret_cast<const float4*>(Cn);
    const int n4 = (B * B) >> 2, b4 = B >> 2;
    constexpr int kBatch = 8;
    for (int f0 = threadIdx.x; f0 < n4; f0 += blockDim.x * kBatch) {
      float4 v[kBatch];
#pragma unroll
      for (int u = 0; u < kBatch; ++u) {
        const int f = f0 + u * blockDim.x;
        if (f < n4) v[u] = C4[f];
      }
#pragma unroll
      for (int u = 0; u < kBatch; ++u) {
        const int f = f0 + u * blockDim.x;
        if (f < n4) {
          const int row = f / b4, col = (f - row * b4) << 2;
          *reinterpret_cast<float4*>(tile + row * PS + col) = v[u];
        }
      }
    }
  }
  __syncthreads();
  float mn = kBig;
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    const int j = q * EPT + e;
    Cr[e] = (i < B && j < B) ? tile[i * PS + j] : kBig;
    Cc[e] = (i < B && j < B) ? tile[j * PS + i] : kBig;
    mn = fminf(mn, Cr[e]);
  }
  const float c0 = block_reduce(mn, red, true);             // (contains the barrier that frees the tile)
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    Cr[e] = (Cr[e] < kBig) ? (Cr[e] - c0) * kscale : kBig;
    Cc[e] = (Cc[e] < kBig) ? (Cc[e] - c0) * kscale : kBig;
  }
  return c0;
}

// log-domain half update of one row (column): ahat - LSE2_e(pot[e] - Cs[e]) over the 4-thread group
template <int EPT>
__device__ __forceinline__ float lse_update(const float (&Cs)[EPT], const float* pot, float ahat) {
  float t[EPT];
  float m = -kBig;
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    t[e] = (Cs[e] < kBig) ? pot[e] - Cs[e] : -kBig;      // padded entries: their potentials are unset
    m = fmaxf(m, t[e]);
  }
  m = group_max<lpr_of(EPT)>(m);
  float s0 = 0.f, s1 = 0.f;
#pragma unroll
  for (int e = 0; e < EPT; e += 2) {
    s0 += fast_exp2(t[e] - m);
    s1 += fast_exp2(t[e + 1] - m);
  }
  return ahat - (m + fast_log2(group_sum<lpr_of(EPT)>(s0 + s1)));
}

// Vectors that every thread reads a 16-element slice of are stored PADDED: chunk q starts at
// q*(EPT+4) floats, so the four chunk addresses of a quarter-warp fall into distinct bank groups
// (an unpadded 64-byte chunk stride makes chunks 0/2 and 1/3 collide: 2-way conflict on every load).
template <int EPT>
__device__ __forceinline__ int pad_index(int j) { return (j / EPT) * (EPT + 4) + (j % EPT); }

// Pins a shared-window address in a register.  Without this ptxas rematerialises the address inside
// the iteration loop from S2R SR_CgaCtaId, whose latency (~200 cycles) then sits in front of the
// mat-vec's loads every half-iteration (measured: 390 -> 510 ns per iteration).
__device__ __forceinline__ uint32_t pin_u32(uint32_t v) {
  uint32_t r;
  asm volatile("mov.u32 %0, %1;" : "=r"(r) : "r"(v));
  return r;
}

__device__ __forceinline__ int lds_flag(uint32_t saddr) {
  int v;
  asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(v) : "r"(saddr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_flag(uint32_t saddr, int v) {
  asm volatile("st.volatile.shared.s32 [%0], %1;" ::"r"(saddr), "r"(v) : "memory");
}

__device__ __forceinline__ void sts128(uint32_t saddr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float lds_f32(uint32_t saddr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(saddr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_f32(uint32_t saddr, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(saddr), "f"(v) : "memory");
}

__device__ __forceinline__ float4 lds128(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
  return v;
}

// mat-vec slice: sum_e Ks[e] * vec[e] over the 4-thread group (4 independent FMA chains);
// `saddr` = shared-window byte address of this thread's (padded) chunk
template <int EPT>
__device__ __forceinline__ float dot_slice(const float (&Ks)[EPT], uint32_t saddr) {
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
  for (int e = 0; e < EPT; e += 4) {
    const float4 b = lds128(saddr + e * 4);
    s0 = fmaf(Ks[e], b.x, s0);
    s1 = fmaf(Ks[e + 1], b.y, s1);
    s2 = fmaf(Ks[e + 2], b.z, s2);
    s3 = fmaf(Ks[e + 3], b.w, s3);
  }
  return group_sum<lpr_of(EPT)>((s0 + s1) + (s2 + s3));
}
}  // namespace

// HS = true: the potential history (L+1 rows of u and v) lives in shared memory during the solve and
// is written to global memory once at the end; HS = false (history too large): one global store per
// half-iteration.
template <int EPT, bool HS>
__global__ void __launch_bounds__(lpr_of(EPT) * lpr_of(EPT) * EPT) sinkhorn_fwd_small_kernel(
    const float* __restrict__ C, int B, float eps, int L, int Lmin, float thresh, int exit_on_index,
    float* __restrict__ u_hist, float* __restrict__ v_hist, int32_t* __restrict__ nits_out,
    float* __restrict__ cost_out, SinkhornMix mix) {
  constexpr int LPR = lpr_of(EPT);
  constexpr int BM = LPR * EPT;
  constexpr int BMP = LPR * (EPT + 4);
  extern __shared__ __align__(16) float hist[];         // HS: Uh[L+1][BM] | Vh[L+1][BM]
  __shared__ __align__(16) float us[BM], vs[BM];        // !HS: current log2-domain potentials
  __shared__ __align__(16) float as[BMP], bs[BMP];      // linear scalings a_i, b_j of the fast path (padded)
  __shared__ float red[32];
  __shared__ int stop_flag, bad_flag;
  // range-guard flags of the post-`first_check` loop, one per iteration parity: iteration `it` writes bad2[it & 1]
  // and iteration it + 1 reads it, so a read and the next write of the same word are always two barriers apart
  // (a single flag let a fast warp's write of iteration it race with a slow warp's read at the top of it)
  __shared__ int bad2[2];
  const int n = blockIdx.x;
  const int tid = threadIdx.x, i = tid / LPR, q = tid % LPR;
  const int ic = min(i, BM - 1);
  const bool owner = (q == 0) && (i < B);
  const float kscale = kLog2e / eps;
  const float ahat = -log2f((float)B);
  const float two_ahat = 1.f / (float)B;
  float Cr[EPT], Cc[EPT], Kr[EPT], Kc[EPT];
  pdl_wait();                    // C comes from the kernel before (cost_finalize_kernel in the fused path)
  pdl_launch_dependents();       // the backward kernel may load its cost slices while this one iterates
  const float* Cn = C + (long long)n * B * B;
  const bool via_tile = HS && (B & 3) == 0 && (reinterpret_cast<uintptr_t>(Cn) & 15) == 0;
  const float c0 = via_tile ? load_slices_tile<EPT>(Cn, B, kscale, red, Cr, Cc, hist)      // the history region is still free
                            : load_slices<EPT>(Cn, B, kscale, red, Cr, Cc);
  float* uh = u_hist + (long long)n * (L + 1) * B;
  float* vh = v_hist + (long long)n * (L + 1) * B;
  float* Uh = hist;
  float* Vh = hist + (HS ? (size_t)(L + 1) * BM : 0);
  // row k of the potentials: smem history (HS) or the single current row (!HS)
  auto urow = [&](int k) -> float* { return HS ? Uh + (size_t)k * BM : us; };
  auto vrow = [&](int k) -> float* { return HS ? Vh + (size_t)k * BM : vs; };

  // absorb the kernel at alpha_i = min_j Chat_ij, beta = 0
  float alpha;
  {
    float rm = kBig;
#pragma unroll
    for (int e = 0; e < EPT; ++e) rm = fminf(rm, Cr[e]);
    alpha = group_min<LPR>(rm);
  }
  const int ip = pad_index<EPT>(ic);                            // padded slot of row / column i
  const uint32_t as_q = pin_u32(static_cast<uint32_t>(__cvta_generic_to_shared(as)) + q * (EPT + 4) * 4);
  const uint32_t bs_q = pin_u32(static_cast<uint32_t>(__cvta_generic_to_shared(bs)) + q * (EPT + 4) * 4);
  const uint32_t bs_i = pin_u32(static_cast<uint32_t>(__cvta_generic_to_shared(&bs[ip])));
  const uint32_t bad_a = pin_u32(static_cast<uint32_t>(__cvta_generic_to_shared(&bad_flag)));
  for (int t = tid; t < BM; t += blockDim.x) { urow(0)[t] = 0.f; vrow(0)[t] = 0.f; }
  for (int t = tid; t < BMP; t += blockDim.x) { as[t] = 0.f; bs[t] = 0.f; }
  if (!HS && tid < B) { uh[tid] = 0.f; vh[tid] = 0.f; }
  if (tid == 0) { stop_flag = 0; bad_flag = 0; bad2[0] = 0; bad2[1] = 0; }
  __syncthreads();
  if (owner) { as[ip] = alpha; bs[ip] = 1.f; }   // stage the row minima for the column slices; b = exp2(0)
  __syncthreads();
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    Kr[e] = fast_exp2(alpha - Cr[e]);                       // padded entries: exp2(x - kBig) = 0
    Kc[e] = fast_exp2(as[q * (EPT + 4) + e] - Cc[e]);
  }
  __syncthreads();
  for (int t = tid; t < BMP; t += blockDim.x) as[t] = 0.f;
  __syncthreads();

  const float ahat_alpha = ahat + alpha;
  float u_cur = 0.f;            // uhat of this thread's row (all four lanes of a row hold it)
  bool slow = false;
  int it = 0, nits = 0;
  // iterations before `first_check` can never stop (gan_utils.py:159 needs nits >= Lmin, :116 needs the
  // index >= Lmin; the last iteration needs no test): they run in a tight loop without the bookkeeping
  const int first_check = min(L - 1, exit_on_index ? Lmin : Lmin - 1);
  for (;;) {
    if (!slow) {
      // Fixed-point short cut: the iteration is a deterministic function of the column scalings b, so
      // once an iteration returns b bit-for-bit (fp32 Sinkhorn does: after 1 iteration on the
      // diagonal-dominant xx / yy problems, after 55-70 on cfg2's uniform xy problem) every later
      // iteration reproduces the same potentials; the remaining history rows are copies.  Only every
      // 8th iteration carries the test (a reducing barrier in place of the plain one); the other seven
      // run in an inner loop with nothing but the two mat-vecs between barriers (a per-iteration test,
      // even off the critical path, cost 65-120 ns of the ~390 ns iteration in control instructions).
      // The range guard rides on the same barrier: plain iterations carry no test at all (inf / NaN from a
      // scaling that left the fp32 range are sticky, so the next tested iteration sees them); a failed test
      // rolls back to the last tested iteration and redoes the block in the log domain.  (A flag load +
      // branch in every iteration was ~40 cycles on the critical path: the bare loop of
      // scripts/matvec_probe.py runs in 569 cycles, this one ran in 800.)
      // Returns 0: continue, 1: a scaling left the safe range, 2: fixed point reached.
      float unew = 0.f, vnew = 0.f;
      auto iteration = [&](auto check_tag) -> int {
        constexpr bool kCheck = decltype(check_tag)::value;
        const float s = dot_slice<EPT>(Kr, bs_q);
        const float a_new = two_ahat * fast_rcp(s);       // critical path first
        unew = ahat + alpha - fast_log2(s);
        if (owner) {
          as[ip] = a_new;
          urow(it + 1)[i] = unew;
          if (!HS) uh[(long long)(it + 1) * B + i] = unew;
        }
        __syncthreads();
        const float t = dot_slice<EPT>(Kc, as_q);
        const float b_new = two_ahat * fast_rcp(t);
        vnew = ahat - fast_log2(t);
        float b_old = 0.f;
        if (kCheck) b_old = lds_f32(bs_i);                // previous b (read before the owner lane's store)
        if (owner) {
          bs[ip] = b_new;
          vrow(it + 1)[i] = vnew;
          if (!HS) vh[(long long)(it + 1) * B + i] = vnew;
          if (kCheck && !(s > kLo && s < kHi && t > kLo && t < kHi)) sts_flag(bad_a, 1);
        }
        if (!kCheck) {
          __syncthreads();
          return 0;
        }
        // (__syncthreads_or returns a truth value, not the OR of the arguments: the rare range failure goes
        //  through the shared flag, the fixed-point vote through the barrier)
        const int fixed = __syncthreads_and((i >= B) | (b_new == b_old));
        if (lds_flag(bad_a) != 0) return 1;
        return fixed ? 2 : 0;
      };
      while (it < first_check) {
        const int block_start = it;
        const int plain_end = it + min(first_check - it, 8) - 1;
        for (; it < plain_end; ++it) iteration(std::false_type{});
        const int rc = iteration(std::true_type{});
        if (rc == 1) {                                    // redo this block of iterations in the log domain
          it = block_start + 1;
          break;
        }
        if (rc == 2) {                                    // rows >= it + 1 are all equal
          if (owner)
            for (int r = it + 2; r <= first_check; ++r) {
              if (HS) { urow(r)[i] = unew; vrow(r)[i] = vnew; }
              else { uh[(long long)r * B + i] = unew; vh[(long long)r * B + i] = vnew; }
            }
          it = first_check;
          break;
        }
        ++it;
      }
      nits = it;
      if (bad_flag) {                                     // iteration it-1 left the safe range: redo it in the log domain
        slow = true;
        it = max(it - 1, 0);
        __syncthreads();
        if (!HS && tid < B) { us[tid] = uh[(long long)it * B + tid]; vs[tid] = vh[(long long)it * B + tid]; }
        __syncthreads();
      } else if (!HS && owner) {
        us[i] = uh[(long long)it * B + i];                // the tight loop does not maintain us / vs
        vs[i] = vh[(long long)it * B + i];
      }
      __syncthreads();
      u_cur = urow(it)[ic];
    }
    while (it < L) {
      float du;
      if (!slow) {
        // ---- fast u update: s_i = sum_j Kt_ij b_j (straight-line; only the stores are predicated)
        const float s = dot_slice<EPT>(Kr, bs_q);
        if (bad2[(it + 1) & 1]) {
          // a scaling left the safe range during iteration it-1: roll back to the potentials before
          // it (history row it-1) and redo it in the log domain
          slow = true;
          --it;
          __syncthreads();
          if (!HS && tid < B) { us[tid] = uh[(long long)it * B + tid]; vs[tid] = vh[(long long)it * B + tid]; }
          __syncthreads();
          u_cur = urow(it)[ic];
          continue;
        }
        const float unew = ahat_alpha - fast_log2(s);
        const float a = two_ahat * fast_rcp(s);
        du = fabsf(unew - u_cur);
        u_cur = unew;
        if (owner) {
          as[ip] = a;
          urow(it + 1)[i] = unew;
          if (!HS) uh[(long long)(it + 1) * B + i] = unew;
          if (!(s > kLo && s < kHi)) bad2[it & 1] = 1;
        }
        __syncthreads();
        // ---- fast v update: t_j = sum_i Kt_ij a_i -------------------------------------------
        const float t = dot_slice<EPT>(Kc, as_q);
        const float vnew = ahat - fast_log2(t);
        const float bnew = two_ahat * fast_rcp(t);
        if (owner) {
          bs[ip] = bnew;
          vrow(it + 1)[i] = vnew;
          if (!HS) vh[(long long)(it + 1) * B + i] = vnew;
          if (!(t > kLo && t < kHi)) bad2[it & 1] = 1;
        }
        __syncthreads();
      } else {
        // ---- log-domain updates (reference formulation) -------------------------------------
        const float unew = lse_update<EPT>(Cr, vrow(it) + q * EPT, ahat);
        du = fabsf(unew - u_cur);
        u_cur = unew;
        if (owner) {
          urow(it + 1)[i] = unew;
          if (!HS) uh[(long long)(it + 1) * B + i] = unew;
        }
        __syncthreads();
        const float vnew = lse_update<EPT>(Cc, urow(it + 1) + q * EPT, ahat);
        if (owner) {
          vrow(it + 1)[i] = vnew;
          if (!HS) vh[(long long)(it + 1) * B + i] = vnew;
        }
        __syncthreads();
      }
      nits = it + 1;
      // ---- stopping rule (gan_utils.py:157-160 / :114-117); can only fire once the minimum count
      // is reached, so the reduction is skipped before that -------------------------------------
      const bool may_stop = exit_on_index ? (it >= Lmin) : (nits >= Lmin);
      if (may_stop && nits < L && (slow || !bad2[it & 1])) {
        const float err = block_reduce(owner ? du : 0.f, red, false) / kscale;
        if (tid == 0) stop_flag = (thresh > err) ? 1 : 0;
        __syncthreads();
        if (stop_flag) break;
      }
      ++it;
    }
    // the last executed iteration may itself have tripped the guard
    if (!slow && nits > 0 && bad2[(nits - 1) & 1]) {
      slow = true;
      it = nits - 1;
      __syncthreads();
      if (!HS && tid < B) { us[tid] = uh[(long long)it * B + tid]; vs[tid] = vh[(long long)it * B + tid]; }
      if (tid == 0) stop_flag = 0;
      __syncthreads();
      u_cur = urow(it)[ic];
      continue;
    }
    break;
  }
  // ---- sharp cost sum(pi * C) ---------------------------------------------------------------
  float s1 = 0.f, s0 = 0.f;
  {
    const float* vfin = vrow(nits) + q * EPT;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const float pi = (Cr[e] < kBig) ? fast_exp2(u_cur + vfin[e] - Cr[e]) : 0.f;
      s0 += pi;
      s1 = fmaf(pi, Cr[e], s1);
    }
    if (i >= B) { s0 = 0.f; s1 = 0.f; }
  }
  s1 = block_reduce(s1, red, false);
  s0 = block_reduce(s0, red, false);
  if (tid == 0) {
    cost_out[n] = s1 / kscale + c0 * s0;
    nits_out[n] = nits;
    if (mix.loss != nullptr) {                          // last CTA of the triple combines the three terms
      __threadfence();
      const int p = n / 3;
      if (atomicAdd(&mix.counter[p], 1) == 2) {
        __threadfence();
        const volatile float* cv = cost_out + 3 * p;
        const float xy = cv[0], xx = cv[1], yy = cv[2];
        mix.loss[p] = 2.f * xy - xx - yy;               // gan_utils.py:225
        if (mix.terms) { mix.terms[3 * p] = xy; mix.terms[3 * p + 1] = xx; mix.terms[3 * p + 2] = yy; }
      }
    }
  }
  if (HS) {
    const int total = (nits + 1) * B;
    if (B == BM && ((reinterpret_cast<uintptr_t>(uh) | reinterpret_cast<uintptr_t>(vh)) & 15) == 0) {
      // rows are contiguous in both places: a straight 16-byte copy, no index arithmetic
      const float4* U4 = reinterpret_cast<const float4*>(Uh);
      const float4* V4 = reinterpret_cast<const float4*>(Vh);
      float4* u4 = reinterpret_cast<float4*>(uh);
      float4* v4 = reinterpret_cast<float4*>(vh);
      for (int f = tid; f < (total >> 2); f += blockDim.x) {
        u4[f] = U4[f];
        v4[f] = V4[f];
      }
    } else {
      for (int k = tid / BM; k <= nits; k += blockDim.x / BM) {
        const int j = tid % BM;
        if (j < B) {
          uh[(long long)k * B + j] = Uh[(size_t)k * BM + j];
          vh[(long long)k * B + j] = Vh[(size_t)k * BM + j];
        }
      }
    }
  }
}

// HS = true: the whole potential history (nits+1 rows of u and v) is copied to shared memory up
// front (51 KB at B=64, L=100) so every step reads its operands with LDS; HS = false (history too
// large): two rows are staged per step with a register prefetch from L2.
// MINB = 2 (launches with more problems than SMs, BASELINE config 4): the register allocation is capped so that two
// CTAs share an SM — the loop is a latency chain, a second CTA fills its bubbles (5.2 waves of one CTA per SM otherwise).
template <int EPT, bool HS, int MINB>
__global__ void __launch_bounds__(lpr_of(EPT) * lpr_of(EPT) * EPT, MINB) sinkhorn_bwd_small_kernel(
    const float* __restrict__ C, int B, float eps, int L, const float* __restrict__ u_hist,
    const float* __restrict__ v_hist, const int32_t* __restrict__ nits_in, const float* __restrict__ gcost,
    float* __restrict__ Cbar, const int32_t* __restrict__ only_if, SinkhornMix mix) {
  if (only_if != nullptr && only_if[blockIdx.x] == 0) return;     // fallback launch: only the declined problems
  constexpr int LPR = lpr_of(EPT);
  constexpr int BM = LPR * EPT;
  constexpr int PQ = EPT + 4;                           // padded chunk stride (see pad_index)
  constexpr int BMP = LPR * PQ;
  extern __shared__ __align__(16) float hist[];         // HS: Uh[nits+1][BMP] | Vh[nits+1][BMP]
  __shared__ __align__(16) float Us[2][BMP], Vs[2][BMP];  // !HS: staged u^k / v^k, v^{k-1}
  __shared__ __align__(16) float un_s[BMP], vn_s[BMP];  // final potentials (absorption reference)
  __shared__ __align__(16) float ub[BMP], vb[BMP];      // adjoints ubar, vbar (slow-path operands)
  __shared__ __align__(16) float ga[BMP], gb[BMP];      // fast path: factor * adjoint vectors
  __shared__ float red[32];
  __shared__ int slow_flag, k_slow;
  const int n = blockIdx.x;
  const int tid = threadIdx.x, i = tid / LPR, q = tid % LPR;
  const bool owner = (q == 0) && (i < B);
  const int ip = pad_index<EPT>(min(i, BM - 1));        // padded slot of row / column i
  const int tp = pad_index<EPT>(min(tid, BM - 1));      // padded slot of element tid (loader threads)
  const int qo = q * PQ;                                // start of this thread's chunk
  const float kscale = kLog2e / eps;
  const float ahat = -log2f((float)B);
  float Cr[EPT], Cc[EPT], Kr[EPT], Kc[EPT], Gr[EPT], Gc[EPT];
  load_slices<EPT>(C + (long long)n * B * B, B, kscale, red, Cr, Cc);   // C predates the forward kernel: safe before the wait
  pdl_wait();                    // history, nits, upstream gradient come from the kernels before
  pdl_launch_dependents();       // the gradient GEMM may start streaming the videos now
  const float* uh = u_hist + (long long)n * (L + 1) * B;
  const float* vh = v_hist + (long long)n * (L + 1) * B;
  const int nits = nits_in[n];
  const float g = mix.gloss ? mix.gloss[n / 3] * ((n % 3 == 0) ? 2.f : -1.f) : gcost[n];
  float* Uh = hist;
  float* Vh = hist + (HS ? (size_t)(nits + 1) * BMP : 0);

  for (int t = tid; t < 2 * BMP; t += blockDim.x) { (&Us[0][0])[t] = 0.f; (&Vs[0][0])[t] = 0.f; }
  for (int t = tid; t < BMP; t += blockDim.x) {
    ub[t] = 0.f; vb[t] = 0.f; ga[t] = 0.f; gb[t] = 0.f; un_s[t] = 0.f; vn_s[t] = 0.f;
  }
  if (tid == 0) { slow_flag = 0; k_slow = -1; }
  __syncthreads();
  if (tid < B) {
    un_s[tp] = uh[(long long)nits * B + tid];
    vn_s[tp] = vh[(long long)nits * B + tid];
  }
  __syncthreads();
  if (HS) {
    // copy the history; remember the last step whose potentials are further than 2^60 from the
    // absorption reference (steps k <= k_slow + 1 use direct exponentials).  All loads of a thread are
    // issued before the first use: the copy is one L2 round trip, not one per element (the element-wise
    // loop was 24 % of the kernel in the ncu source view, profiles/r1_ncu_summary.md).
    const int total = (nits + 1) * B;
    int kmax = -1;
    if (B < BM) {                                       // padded columns are read (times zero weights): keep them finite
      for (int e = tid; e < 2 * (nits + 1) * BMP; e += blockDim.x) hist[e] = 0.f;
      __syncthreads();
    }
    if ((B & 3) == 0 && ((reinterpret_cast<uintptr_t>(uh) | reinterpret_cast<uintptr_t>(vh)) & 15) == 0) {
      const float4* u4 = reinterpret_cast<const float4*>(uh);
      const float4* v4 = reinterpret_cast<const float4*>(vh);
      auto sa = [](const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); };
      const uint32_t un_a = pin_u32(sa(un_s)), vn_a = pin_u32(sa(vn_s));
      const uint32_t U_a = pin_u32(sa(Uh)), V_a = pin_u32(sa(Vh));
      const int B4 = B >> 2;
      constexpr int kBatch = 8;
      for (int f0 = tid; f0 < (total >> 2); f0 += blockDim.x * kBatch) {
        float4 u[kBatch], v[kBatch];
#pragma unroll
        for (int t = 0; t < kBatch; ++t) {
          const int f = f0 + t * blockDim.x;
          if (f < (total >> 2)) { u[t] = u4[f]; v[t] = v4[f]; }
        }
#pragma unroll
        for (int t = 0; t < kBatch; ++t) {
          const int f = f0 + t * blockDim.x;
          if (f < (total >> 2)) {
            const int k = f / B4, j = (f - k * B4) << 2;
            const uint32_t jp = (uint32_t)pad_index<EPT>(j) * 4;   // 4 consecutive columns stay inside one chunk
            const float4 ru = lds128(un_a + jp);
            const float4 rv = lds128(vn_a + jp);
            const bool ok = fabsf(u[t].x - ru.x) <= kExpLim && fabsf(u[t].y - ru.y) <= kExpLim &&
                            fabsf(u[t].z - ru.z) <= kExpLim && fabsf(u[t].w - ru.w) <= kExpLim &&
                            fabsf(v[t].x - rv.x) <= kExpLim && fabsf(v[t].y - rv.y) <= kExpLim &&
                            fabsf(v[t].z - rv.z) <= kExpLim && fabsf(v[t].w - rv.w) <= kExpLim;
            if (!ok) kmax = max(kmax, k);
            sts128(U_a + (uint32_t)k * (BMP * 4) + jp, u[t]);
            sts128(V_a + (uint32_t)k * (BMP * 4) + jp, v[t]);
          }
        }
      }
    } else {
      constexpr int kBatch = 8;
      for (int e0 = tid; e0 < total; e0 += blockDim.x * kBatch) {
        float u[kBatch], v[kBatch];
#pragma unroll
        for (int t = 0; t < kBatch; ++t) {
          const int e = e0 + t * blockDim.x;
          if (e < total) { u[t] = uh[e]; v[t] = vh[e]; }
        }
#pragma unroll
        for (int t = 0; t < kBatch; ++t) {
          const int e = e0 + t * blockDim.x;
          if (e < total) {
            const int k = e / B, j = e - k * B;
            const int jp = pad_index<EPT>(j);
            if (!(fabsf(u[t] - un_s[jp]) <= kExpLim) || !(fabsf(v[t] - vn_s[jp]) <= kExpLim)) kmax = max(kmax, k);
            Uh[(size_t)k * BMP + jp] = u[t];
            Vh[(size_t)k * BMP + jp] = v[t];
          }
        }
      }
    }
    if (kmax >= 0) atomicMax(&k_slow, kmax);
  } else if (tid < B) {
    Us[nits & 1][tp] = un_s[tp];
    Vs[nits & 1][tp] = vn_s[tp];
    if (nits >= 1) {
      const float vm = vh[(long long)(nits - 1) * B + tid];
      Vs[(nits - 1) & 1][tp] = vm;
      if (!(fabsf(vm - vn_s[tp]) <= kExpLim)) slow_flag = 1;
    }
  }
  __syncthreads();
  const float un_i = un_s[ip], vn_i = vn_s[ip];    // row i / column i of this thread
  // ---- adjoint seeds.  cost = sum(pi*C) = sum(pi*(C - c0)) + c0*sum(pi), and sum(pi) == 1 identically
  // in the inputs (the last v-update normalises every column of pi to 1/B), so the c0 term has zero
  // gradient: seed with C' = C - c0.  Cbar = pi (1 - C'/eps), ubar = rowsum(pi C')/eps, vbar =
  // colsum(pi C')/eps.  This removes the O(|C|/eps) cancellation the reference's fp32 gradient suffers.
  {
    float ru = 0.f, rv = 0.f;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const float ce_r = Cr[e] * kLn2;                              // (C - c0) / eps (row slice)
      Kr[e] = fast_exp2(un_i + vn_s[qo + e] - Cr[e]);               // pi, row slice
      Gr[e] = Kr[e] * (1.f - ce_r);
      ru = fmaf(Kr[e], ce_r, ru);
      const float ce_c = Cc[e] * kLn2;
      Kc[e] = fast_exp2(un_s[qo + e] + vn_i - Cc[e]);               // pi, column slice
      rv = fmaf(Kc[e], ce_c, rv);
      Gc[e] = 0.f;
    }
    ru = group_sum<LPR>(ru);
    rv = group_sum<LPR>(rv);
    if (owner) {
      ub[ip] = ru;
      vb[ip] = rv;
      gb[ip] = (float)B * rv;          // exp2(v^n_j - v^n_j - ahat) * vbar_j
    }
  }
  __syncthreads();
  const uint32_t ga_q = pin_u32(static_cast<uint32_t>(__cvta_generic_to_shared(ga)) + qo * 4);
  const uint32_t gb_q = pin_u32(static_cast<uint32_t>(__cvta_generic_to_shared(gb)) + qo * 4);
  const int kslow = HS ? k_slow : -1;
  // pinned shared-window addresses of this thread's elements (see pin_u32)
  auto sa = [](const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); };
  const uint32_t ub_i = pin_u32(sa(&ub[ip])), vb_i = pin_u32(sa(&vb[ip]));
  const uint32_t ga_i = pin_u32(sa(&ga[ip])), gb_i = pin_u32(sa(&gb[ip]));
  const uint32_t Uh_i = pin_u32(sa(HS ? &Uh[ip] : &Us[0][ip])), Vh_i = pin_u32(sa(HS ? &Vh[ip] : &Vs[0][ip]));

  int k = nits;
  if (HS) {
    // ---- fast steps (all potentials within 2^60 of the absorption reference): a loop with nothing but
    // the two mat-vecs, the rank-one accumulation and two barriers; every branch removed from it was
    // worth 10-20 ns of the ~420 ns step (single-warp-per-scheduler latency, see the forward kernel).
    float ub_carry = owner ? lds_f32(ub_i) : 0.f;        // the seed enters the first step only
    const uint32_t step_bytes = BMP * 4;
    uint32_t u_a = Uh_i + (uint32_t)k * step_bytes, v_a = Vh_i + (uint32_t)(k - 1) * step_bytes;
    for (; k >= max(kslow + 2, 1); --k, u_a -= step_bytes, v_a -= step_bytes) {
      const float uk_i = lds_f32(u_a);
      const float fa = fast_exp2(uk_i - un_i);
      float a0 = 0.f, a1 = 0.f;
#pragma unroll
      for (int e = 0; e < EPT; e += 4) {
        const float4 w = lds128(gb_q + e * 4);
        const float t0 = Kr[e] * w.x, t1 = Kr[e + 1] * w.y, t2 = Kr[e + 2] * w.z, t3 = Kr[e + 3] * w.w;
        Gr[e] = fmaf(t0, fa, Gr[e]);
        Gr[e + 1] = fmaf(t1, fa, Gr[e + 1]);
        Gr[e + 2] = fmaf(t2, fa, Gr[e + 2]);
        Gr[e + 3] = fmaf(t3, fa, Gr[e + 3]);
        a0 += t0 + t2;
        a1 += t1 + t3;
      }
      const float ubn = ub_carry - group_sum<LPR>((a0 + a1) * fa);
      ub_carry = 0.f;
      if (owner) {
        sts_f32(ub_i, ubn);
        sts_f32(ga_i, fa * ubn);                          // |u^k - u^n| <= 2^60 here: no clamp needed
      }
      __syncthreads();
      const float vkm1_j = lds_f32(v_a);
      const float fb = fast_exp2(vkm1_j - vn_i - ahat);
      float c0 = 0.f, c1 = 0.f;
#pragma unroll
      for (int e = 0; e < EPT; e += 4) {
        const float4 w = lds128(ga_q + e * 4);
        const float t0 = Kc[e] * w.x, t1 = Kc[e + 1] * w.y, t2 = Kc[e + 2] * w.z, t3 = Kc[e + 3] * w.w;
        Gc[e] = fmaf(t0, fb, Gc[e]);
        Gc[e + 1] = fmaf(t1, fb, Gc[e + 1]);
        Gc[e + 2] = fmaf(t2, fb, Gc[e + 2]);
        Gc[e + 3] = fmaf(t3, fb, Gc[e + 3]);
        c0 += t0 + t2;
        c1 += t1 + t3;
      }
      const float vbn = -group_sum<LPR>((c0 + c1) * fb);
      if (owner) {
        sts_f32(vb_i, vbn);
        sts_f32(gb_i, fb * vbn);
      }
      __syncthreads();
    }
  }
  bool slow = false;
  for (; k >= 1; --k) {
    const int b = k & 1;
    const float* Uk = HS ? Uh + (size_t)k * BMP : Us[b];
    const float* Vk = HS ? Vh + (size_t)k * BMP : Vs[b];
    const float* Vkm1 = HS ? Vh + (size_t)(k - 1) * BMP : Vs[b ^ 1];
    // !HS: prefetch the next step's potentials (L2) while this step computes
    float pu = 0.f, pv = 0.f;
    if (!HS && tid < B && k >= 2) {
      pu = uh[(long long)(k - 1) * B + tid];
      pv = vh[(long long)(k - 2) * B + tid];
    }
    if (HS) slow = (k <= kslow + 1);
    else if (!slow) slow = (slow_flag != 0);
    // ---- through v^k = a - eps*LSE_i((u^k_i - C_ij)/eps):  Pv_ij = exp((u^k_i + v^k_j - a - C_ij)/eps)
    //      Cbar += Pv * vbar_j ;  ubar_i = (k == nits ? ubar_i : 0) - sum_j Pv_ij vbar_j
    {
      const float uk_i = lds_f32(Uh_i + (HS ? k : b) * (BMP * 4));
      float part;
      if (!slow) {
        // Pv_ij vbar_j = pi_ij * exp2(u^k_i - u^n_i) * gb_j
        const float fa = fast_exp2(uk_i - un_i);
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int e = 0; e < EPT; e += 4) {
          const float4 w = lds128(gb_q + e * 4);
          const float t0 = Kr[e] * w.x, t1 = Kr[e + 1] * w.y, t2 = Kr[e + 2] * w.z, t3 = Kr[e + 3] * w.w;
          Gr[e] = fmaf(t0, fa, Gr[e]);
          Gr[e + 1] = fmaf(t1, fa, Gr[e + 1]);
          Gr[e + 2] = fmaf(t2, fa, Gr[e + 2]);
          Gr[e + 3] = fmaf(t3, fa, Gr[e + 3]);
          a0 += t0 + t2;
          a1 += t1 + t3;
        }
        part = (a0 + a1) * fa;
      } else {
        const float ui = uk_i - ahat;
        float a0 = 0.f;
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
          const float w = fast_exp2(ui + Vk[qo + e] - Cr[e]) * vb[qo + e];
          Gr[e] += w;
          a0 += w;
        }
        part = a0;
      }
      const float acc = group_sum<LPR>(part);
      if (owner) {
        const float ubn = ((k == nits) ? lds_f32(ub_i) : 0.f) - acc;
        sts_f32(ub_i, ubn);
        sts_f32(ga_i, fast_exp2(fminf(fmaxf(uk_i - un_i, -kExpLim), kExpLim)) * ubn);   // for the column phase
      }
    }
    __syncthreads();
    if (!HS && !slow) slow = (slow_flag != 0);
    // ---- through u^k = a - eps*LSE_j((v^{k-1}_j - C_ij)/eps):  Pu_ij = exp((u^k_i + v^{k-1}_j - a - C_ij)/eps)
    //      Cbar += Pu * ubar_i ;  vbar_j = - sum_i Pu_ij ubar_i
    {
      const float vkm1_j = lds_f32(Vh_i + (HS ? k - 1 : (b ^ 1)) * (BMP * 4));
      const float fb = fast_exp2(fminf(fmaxf(vkm1_j - vn_i, -kExpLim), kExpLim) - ahat);
      float part;
      if (!slow) {
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int e = 0; e < EPT; e += 4) {
          const float4 w = lds128(ga_q + e * 4);
          const float t0 = Kc[e] * w.x, t1 = Kc[e + 1] * w.y, t2 = Kc[e + 2] * w.z, t3 = Kc[e + 3] * w.w;
          Gc[e] = fmaf(t0, fb, Gc[e]);
          Gc[e + 1] = fmaf(t1, fb, Gc[e + 1]);
          Gc[e + 2] = fmaf(t2, fb, Gc[e + 2]);
          Gc[e + 3] = fmaf(t3, fb, Gc[e + 3]);
          a0 += t0 + t2;
          a1 += t1 + t3;
        }
        part = (a0 + a1) * fb;
      } else {
        const float vj = vkm1_j - ahat;
        float a0 = 0.f;
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
          const float w = fast_exp2(Uk[qo + e] + vj - Cc[e]) * ub[qo + e];
          Gc[e] += w;
          a0 += w;
        }
        part = a0;
      }
      const float acc = group_sum<LPR>(part);
      if (owner) {
        sts_f32(vb_i, -acc);
        sts_f32(gb_i, fb * (-acc));          // factor of the next row phase: v^{k-1} here is its v^k
      }
      if (!HS && tid < B && k >= 2) {
        Us[b ^ 1][tp] = pu;     // u^{k-1}
        Vs[b][tp] = pv;         // v^{k-2}   (v^k is dead after the row phase above)
        // a potential further than 2^60 from the reference: direct exponentials from the next step on
        if (!(fabsf(pu - un_s[tp]) <= kExpLim) || !(fabsf(pv - vn_s[tp]) <= kExpLim)) slow_flag = 1;
      }
    }
    __syncthreads();
  }
  // ---- Cbar = g * (Gr + Gc^T) ---------------------------------------------------------------
  float* out = Cbar + (long long)n * B * B;
  if (HS) {
    // transpose the column-slice accumulators through shared memory (the history is dead) and write
    // every row once, 16 bytes at a time (the read-modify-write through global memory took 2.9 us)
    constexpr int TS = BM + 1;
    float* T = hist;                                      // launcher guarantees BM * TS floats
#pragma unroll
    for (int e = 0; e < EPT; ++e) T[(q * EPT + e) * TS + min(i, BM - 1)] = Gc[e];
    __syncthreads();
    if (i < B) {
      float o[EPT];
#pragma unroll
      for (int e = 0; e < EPT; ++e) o[e] = g * (Gr[e] + T[i * TS + q * EPT + e]);
      float* dst = out + (long long)i * B + q * EPT;
      if ((B & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
#pragma unroll
        for (int e = 0; e < EPT; e += 4)
          if (q * EPT + e < B) *reinterpret_cast<float4*>(dst + e) = make_float4(o[e], o[e + 1], o[e + 2], o[e + 3]);
      } else {
#pragma unroll
        for (int e = 0; e < EPT; ++e)
          if (q * EPT + e < B) dst[e] = o[e];
      }
    }
  } else {
    if (i < B) {
#pragma unroll
      for (int e = 0; e < EPT; ++e) {
        const int j = q * EPT + e;
        if (j < B) out[(long long)i * B + j] = g * Gr[e];
      }
    }
    __syncthreads();
    if (i < B) {
#pragma unroll
      for (int e = 0; e < EPT; ++e) {
        const int r = q * EPT + e;
        if (r < B) out[(long long)r * B + i] += g * Gc[e];
      }
    }
  }
}

template <int EPT>
static int launch_fwd_t(const float* C, int nsolve, int B, float eps, int L, int Lmin, float thresh, int exit_on_index,
                        float* u_hist, float* v_hist, int32_t* nits, float* cost, int threads, cudaStream_t st, SinkhornMix mix) {
  const size_t hist_bytes = (size_t)2 * (L + 1) * lpr_of(EPT) * EPT * sizeof(float);
  if (hist_bytes <= 160 * 1024) {
    static size_t attr[kMaxDevices] = {};
    if (smem_attr_needed(attr, 160 * 1024))
      KCCOT_CUDA(cudaFuncSetAttribute(sinkhorn_fwd_small_kernel<EPT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)(160 * 1024)));
    const size_t tile_bytes = (size_t)(lpr_of(EPT) * EPT) * (lpr_of(EPT) * EPT + 4) * sizeof(float);   // load_slices_tile
    KCCOT_CUDA(launch_pdl(sinkhorn_fwd_small_kernel<EPT, true>, dim3(nsolve), dim3(threads),
                          hist_bytes > tile_bytes ? hist_bytes : tile_bytes, st, C, B, eps, L, Lmin,
                          thresh, exit_on_index, u_hist, v_hist, nits, cost, mix));
  } else {
    KCCOT_CUDA(launch_pdl(sinkhorn_fwd_small_kernel<EPT, false>, dim3(nsolve), dim3(threads), (size_t)0, st, C, B, eps, L, Lmin,
                          thresh, exit_on_index, u_hist, v_hist, nits, cost, mix));
  }
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}

int launch_sinkhorn_fwd_small(const float* C, int nsolve, int B, float eps, int L, int Lmin, float thresh,
                              int exit_on_index, float* u_hist, float* v_hist, int32_t* nits, float* cost,
                              cudaStream_t st, SinkhornMix mix) {
  const int t4 = ((4 * B + 31) / 32) * 32, t2 = ((2 * B + 31) / 32) * 32;
  if (B <= 32)
    return launch_fwd_t<8>(C, nsolve, B, eps, L, Lmin, thresh, exit_on_index, u_hist, v_hist, nits, cost, t4, st, mix);
  return launch_fwd_t<32>(C, nsolve, B, eps, L, Lmin, thresh, exit_on_index, u_hist, v_hist, nits, cost, t2, st, mix);
}

template <int EPT, int MINB>
static int launch_bwd_t(const float* C, int nsolve, int B, float eps, int L, const float* u_hist, const float* v_hist,
                        const int32_t* nits, const float* gcost, float* Cbar, const int32_t* only_if, int threads,
                        cudaStream_t st, SinkhornMix mix) {
  const size_t hist_bytes = (size_t)2 * (L + 1) * lpr_of(EPT) * (EPT + 4) * sizeof(float);
  if (hist_bytes <= 160 * 1024) {
    static size_t attr[kMaxDevices] = {};
    if (smem_attr_needed(attr, 160 * 1024))
      KCCOT_CUDA(cudaFuncSetAttribute(sinkhorn_bwd_small_kernel<EPT, true, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)(160 * 1024)));
    const size_t tile_bytes = (size_t)(lpr_of(EPT) * EPT) * (lpr_of(EPT) * EPT + 1) * sizeof(float);      // Cbar transposition tile of the epilogue
    KCCOT_CUDA(launch_pdl(sinkhorn_bwd_small_kernel<EPT, true, MINB>, dim3(nsolve), dim3(threads),
                          hist_bytes > tile_bytes ? hist_bytes : tile_bytes, st, C, B, eps, L, u_hist, v_hist, nits, gcost,
                          Cbar, only_if, mix));
  } else {
    KCCOT_CUDA(launch_pdl(sinkhorn_bwd_small_kernel<EPT, false, MINB>, dim3(nsolve), dim3(threads), (size_t)0, st, C, B, eps, L,
                          u_hist, v_hist, nits, gcost, Cbar, only_if, mix));
  }
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}

int launch_sinkhorn_bwd_small(const float* C, int nsolve, int B, float eps, int L, const float* u_hist,
                              const float* v_hist, const int32_t* nits, const float* gcost, float* Cbar,
                              const int32_t* only_if, cudaStream_t st, SinkhornMix mix) {
  // always four lanes per row: the backward carries three times the arithmetic of the forward per element
  // (rank-one accumulation of Cbar), and with two lanes its single warp per scheduler becomes issue-bound
  // (measured: backward chain 72 -> 87 us), while the forward gains (33 -> 28 us)
  const int t4 = ((4 * B + 31) / 32) * 32;
  const bool many = nsolve > num_sms();
  if (B <= 32)
    return many ? launch_bwd_t<8, 2>(C, nsolve, B, eps, L, u_hist, v_hist, nits, gcost, Cbar, only_if, t4, st, mix)
                : launch_bwd_t<8, 0>(C, nsolve, B, eps, L, u_hist, v_hist, nits, gcost, Cbar, only_if, t4, st, mix);
  return many ? launch_bwd_t<16, 2>(C, nsolve, B, eps, L, u_hist, v_hist, nits, gcost, Cbar, only_if, t4, st, mix)
              : launch_bwd_t<16, 0>(C, nsolve, B, eps, L, u_hist, v_hist, nits, gcost, Cbar, only_if, t4, st, mix);
}

}  // namespace kccot
