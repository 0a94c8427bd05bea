// Log-domain Sinkhorn for any B, the fallback of the shapes the other two paths do not take: the
// cost rows are streamed from L2/HBM, one launch per iteration half-pair, so a kernel boundary is
// the grid-wide synchronisation point.  Same internal units as the register-resident path
// (sinkhorn_small.cu): log2 domain, cost shifted by its global minimum.
//
// A CTA owns RC consecutive rows.  Phase 1 (warp per row) does the row reduction, phase 2 (thread
// per column) the column partials over the CTA's rows; partials are combined over CTAs by the
// *_combine kernels.  gan_utils.py:151-164 and SURVEY.md Appendix A.
#include "common.cuh"
#include "sinkhorn.cuh"

namespace kccot {

namespace {
constexpr int RC = 32;     // rows per CTA
constexpr int NT = 256;
constexpr float kNegBig = -3.0e38f;

struct StreamState {
  float shift;      // c0 = min(C)
  float err;        // sum |u - u_prev| of the current iteration (log2 units)
  int done;         // 1 once the stopping rule fired
  int nits;         // executed iterations when done
  float s0, s1;     // sum(pi), sum(pi * Chat) accumulators of the final cost
};

__device__ __forceinline__ void atomic_min_float(float* addr, float v) {
  if (v >= 0.f) atomicMin(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMax(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

__global__ void stream_state_init_kernel(StreamState* s) {
  s->shift = __int_as_float(0x7f800000);
  s->err = 0.f; s->done = 0; s->nits = 0; s->s0 = 0.f; s->s1 = 0.f;
}

__global__ void __launch_bounds__(NT) stream_min_kernel(const float* __restrict__ C, long long n, StreamState* s) {
  float m = 3.0e38f;
  for (long long i = (long long)blockIdx.x * NT + threadIdx.x; i < n; i += (long long)gridDim.x * NT) m = fminf(m, C[i]);
  m = warp_min(m);
  if ((threadIdx.x & 31) == 0) atomic_min_float(&s->shift, m);
}

// online (max, sumexp2) accumulation
__device__ __forceinline__ void lse_push(float t, float& m, float& s) {
  if (t > m) { s = s * fast_exp2(m - t) + 1.f; m = t; }
  else s += fast_exp2(t - m);
}
__device__ __forceinline__ void lse_warp_merge(float& m, float& s) {
  const float M = warp_max(m);
  s = warp_sum(s * fast_exp2(m - M));
  m = M;
}

// One CTA per SM is enough (the grid has B / RC CTAs): without the bound ptxas caps the kernel at 128
// registers and spills part of t[RC].
__global__ void __launch_bounds__(NT, 1) stream_fwd_rows_kernel(const float* __restrict__ C, int B, float kscale,
                                                                float ahat, const float* __restrict__ v_cur,
                                                                float* __restrict__ u_cur,
                                                                float* __restrict__ u_hist_row,
                                                                float* __restrict__ colmax_part,
                                                                float* __restrict__ colsum_part, StreamState* state,
                                                                int track_err) {
  if (state->done) return;
  __shared__ float us[RC];
  const float c0 = state->shift;
  const int r0 = blockIdx.x * RC;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float errw = 0.f;
  for (int rr = warp; rr < RC; rr += NT / 32) {
    const int r = r0 + rr;
    if (r >= B) { if (lane == 0) us[rr] = kNegBig; continue; }
    const float* row = C + (long long)r * B;
    float m = kNegBig, s = 0.f;
    for (int j = lane; j < B; j += 32) lse_push(v_cur[j] - (row[j] - c0) * kscale, m, s);
    lse_warp_merge(m, s);
    const float unew = ahat - (m + fast_log2(s));
    if (lane == 0) {
      if (track_err) errw += fabsf(unew - u_cur[r]);
      us[rr] = unew;
      u_cur[r] = unew;
      if (u_hist_row) u_hist_row[r] = unew;
    }
  }
  if (track_err && lane == 0 && errw != 0.f) atomicAdd(&state->err, errw);
  __syncthreads();
  const int nrows = min(RC, B - r0);
  for (int j = threadIdx.x; j < B; j += NT) {
    float t[RC];
    float m = kNegBig;
#pragma unroll
    for (int rr = 0; rr < RC; ++rr) {
      t[rr] = (rr < nrows) ? us[rr] - (C[(long long)(r0 + rr) * B + j] - c0) * kscale : kNegBig;
      m = fmaxf(m, t[rr]);
    }
    float s = 0.f;
#pragma unroll
    for (int rr = 0; rr < RC; ++rr) s += (rr < nrows) ? fast_exp2(t[rr] - m) : 0.f;
    colmax_part[(long long)blockIdx.x * B + j] = m;
    colsum_part[(long long)blockIdx.x * B + j] = s;
  }
}

__global__ void __launch_bounds__(NT) stream_fwd_combine_kernel(const float* __restrict__ colmax_part,
                                                                const float* __restrict__ colsum_part, int nparts,
                                                                int B, float ahat, float* __restrict__ v_cur,
                                                                float* __restrict__ v_hist_row,
                                                                const StreamState* state) {
  if (state->done) return;
  const int j = blockIdx.x * NT + threadIdx.x;
  if (j >= B) return;
  float M = kNegBig;
  for (int p = 0; p < nparts; ++p) M = fmaxf(M, colmax_part[(long long)p * B + j]);
  float S = 0.f;
  for (int p = 0; p < nparts; ++p) S += colsum_part[(long long)p * B + j] * fast_exp2(colmax_part[(long long)p * B + j] - M);
  const float v = ahat - (M + fast_log2(S));
  v_cur[j] = v;
  if (v_hist_row) v_hist_row[j] = v;
}

__global__ void stream_stop_kernel(StreamState* state, int iter_1based, float thresh, float kscale, int cond_ok) {
  if (state->done) return;
  const float err = state->err / kscale;
  state->err = 0.f;
  if (cond_ok && thresh > err) { state->done = 1; state->nits = iter_1based; }
}

__global__ void __launch_bounds__(NT) stream_cost_kernel(const float* __restrict__ C, int B, float kscale,
                                                         const float* __restrict__ u_cur,
                                                         const float* __restrict__ v_cur, StreamState* state) {
  const float c0 = state->shift;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float s0 = 0.f, s1 = 0.f;
  for (int r = blockIdx.x * (NT / 32) + warp; r < B; r += gridDim.x * (NT / 32)) {
    const float* row = C + (long long)r * B;
    const float ui = u_cur[r];
    for (int j = lane; j < B; j += 32) {
      const float ch = (row[j] - c0) * kscale;
      const float pi = fast_exp2(ui + v_cur[j] - ch);
      s0 += pi;
      s1 = fmaf(pi, ch, s1);
    }
  }
  s0 = warp_sum(s0);
  s1 = warp_sum(s1);
  if (lane == 0) { atomicAdd(&state->s0, s0); atomicAdd(&state->s1, s1); }
}

__global__ void stream_cost_finish_kernel(StreamState* state, float kscale, int L, float* cost, int32_t* nits) {
  if (cost) *cost = state->s1 / kscale + state->shift * state->s0;
  if (nits) *nits = state->done ? state->nits : L;
}

// ------------------------------------ backward ---------------------------------------------------
// seed:  Cbar = g pi (1 - C/eps),  ubar_i = g sum_j pi C/eps,  column partials of g pi C/eps
__global__ void __launch_bounds__(NT) stream_bwd_seed_kernel(const float* __restrict__ C, int B, float kscale,
                                                             float inv_eps,
                                                             const float* __restrict__ u_hist,
                                                             const float* __restrict__ v_hist,
                                                             const int32_t* __restrict__ nits_p,
                                                             const float* __restrict__ gcost,
                                                             const float* __restrict__ shift_p,
                                                             float* __restrict__ Cbar, float* __restrict__ ubar,
                                                             float* __restrict__ colsum_part) {
  __shared__ float us[RC];
  const float shift = *shift_p;
  const int nits = *nits_p;
  const float g = *gcost;
  const float* u = u_hist + (long long)nits * B;
  const float* v = v_hist + (long long)nits * B;
  const int r0 = blockIdx.x * RC;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int rr = warp; rr < RC; rr += NT / 32) {
    const int r = r0 + rr;
    if (r >= B) { if (lane == 0) us[rr] = 0.f; continue; }
    const float* row = C + (long long)r * B;
    float* grow = Cbar + (long long)r * B;
    const float ui = u[r];
    float acc = 0.f;
    for (int j = lane; j < B; j += 32) {
      const float ch = (row[j] - shift) * kscale;
      const float ce = (row[j] - shift) * inv_eps;      // shifted cost: sum(pi) == 1 has zero gradient
      const float pi = g * fast_exp2(ui + v[j] - ch);
      grow[j] = pi * (1.f - ce);
      acc = fmaf(pi, ce, acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) { ubar[r] = acc; us[rr] = ui; }
  }
  __syncthreads();
  const int nrows = min(RC, B - r0);
  for (int j = threadIdx.x; j < B; j += NT) {
    float acc = 0.f;
    const float vj = v[j];
    for (int rr = 0; rr < nrows; ++rr) {
      const float c = C[(long long)(r0 + rr) * B + j];
      acc = fmaf(g * fast_exp2(us[rr] + vj - (c - shift) * kscale), (c - shift) * inv_eps, acc);
    }
    colsum_part[(long long)blockIdx.x * B + j] = acc;
  }
}

// reverse step k:  rows: Pv -> Cbar += Pv*vbar_j, ubar_i = (first ? ubar_i : 0) - sum_j Pv vbar_j
//                  cols: Pu -> Cbar += Pu*ubar_i, partial of sum_i Pu ubar_i
// The operands are located in the saved history by the device-side iteration count.
__global__ void __launch_bounds__(NT) stream_bwd_rows_kernel(const float* __restrict__ C, int B, float kscale, float ahat,
                                                             const float* __restrict__ u_hist,
                                                             const float* __restrict__ v_hist,
                                                             const int32_t* __restrict__ nits_p, int k,
                                                             const float* __restrict__ shift_p,
                                                             const float* __restrict__ vbar, float* __restrict__ ubar,
                                                             float* __restrict__ Cbar,
                                                             float* __restrict__ colsum_part) {
  const int nits = *nits_p;
  if (k > nits) return;
  const float* __restrict__ uk = u_hist + (long long)k * B;
  const float* __restrict__ vk = v_hist + (long long)k * B;
  const float* __restrict__ vkm1 = v_hist + (long long)(k - 1) * B;
  const bool first = k == nits;
  const float shift = *shift_p;
  __shared__ float us[RC], ubs[RC];
  const int r0 = blockIdx.x * RC;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int rr = warp; rr < RC; rr += NT / 32) {
    const int r = r0 + rr;
    if (r >= B) { if (lane == 0) { us[rr] = 0.f; ubs[rr] = 0.f; } continue; }
    const float* row = C + (long long)r * B;
    float* grow = Cbar + (long long)r * B;
    const float ui = uk[r] - ahat;
    float acc = 0.f;
    for (int j = lane; j < B; j += 32) {
      const float w = fast_exp2(ui + vk[j] - (row[j] - shift) * kscale) * vbar[j];
      grow[j] += w;
      acc += w;
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      const float ub = (first ? ubar[r] : 0.f) - acc;
      ubar[r] = ub;
      us[rr] = ui;
      ubs[rr] = ub;
    }
  }
  __syncthreads();
  const int nrows = min(RC, B - r0);
  for (int j = threadIdx.x; j < B; j += NT) {
    float acc = 0.f;
    const float vj = vkm1[j];
    for (int rr = 0; rr < nrows; ++rr) {
      const long long idx = (long long)(r0 + rr) * B + j;
      const float w = fast_exp2(us[rr] + vj - (C[idx] - shift) * kscale) * ubs[rr];
      Cbar[idx] += w;
      acc += w;
    }
    colsum_part[(long long)blockIdx.x * B + j] = acc;
  }
}

__global__ void __launch_bounds__(NT) stream_bwd_combine_kernel(const float* __restrict__ colsum_part, int nparts, int B,
                                                                float sign, float* __restrict__ vbar,
                                                                const int32_t* __restrict__ nits_p, int k) {
  if (nits_p && k > *nits_p) return;
  const int j = blockIdx.x * NT + threadIdx.x;
  if (j >= B) return;
  float acc = 0.f;
  for (int p = 0; p < nparts; ++p) acc += colsum_part[(long long)p * B + j];
  vbar[j] = sign * acc;
}
}  // namespace

// ------------------------------------------------------------------------------------------------
size_t stream_workspace_bytes(int B) {
  const size_t nchunk = (B + RC - 1) / RC;
  return align_up(256 + (size_t)4 * B * 4 + 2 * nchunk * (size_t)B * 4 + 1024, 256);
}

struct StreamWs {
  StreamState* state;
  float *u_cur, *v_cur, *ubar, *vbar, *part_a, *part_b;
  int nchunk;
};
static StreamWs carve(void* ws, int B) {
  StreamWs w;
  char* p = (char*)ws;
  w.state = (StreamState*)p; p += 256;
  w.u_cur = (float*)p; p += (size_t)B * 4;
  w.v_cur = (float*)p; p += (size_t)B * 4;
  w.ubar = (float*)p; p += (size_t)B * 4;
  w.vbar = (float*)p; p += (size_t)B * 4;
  w.nchunk = (B + RC - 1) / RC;
  w.part_a = (float*)p; p += (size_t)w.nchunk * B * 4;
  w.part_b = (float*)p;
  return w;
}

int stream_sinkhorn_fwd(const float* C, int B, float eps, int L, int Lmin, float thresh, int exit_on_index,
                        float* u_hist, float* v_hist, int32_t* nits, float* cost, void* ws, cudaStream_t st) {
  StreamWs w = carve(ws, B);
  const float kscale = kLog2e / eps, ahat = -log2f((float)B);
  stream_state_init_kernel<<<1, 1, 0, st>>>(w.state);
  KCCOT_LAUNCH_CHECK();
  KCCOT_CUDA(cudaMemsetAsync(w.u_cur, 0, (size_t)2 * B * 4, st));          // u_cur, v_cur
  KCCOT_CUDA(cudaMemsetAsync(u_hist, 0, (size_t)B * 4, st));
  KCCOT_CUDA(cudaMemsetAsync(v_hist, 0, (size_t)B * 4, st));
  stream_min_kernel<<<min(4 * num_sms(), (int)(((long long)B * B + NT - 1) / NT)), NT, 0, st>>>(C, (long long)B * B, w.state);
  KCCOT_LAUNCH_CHECK();
  const int cgrid = (B + NT - 1) / NT;
  for (int it = 0; it < L; ++it) {
    const bool may_stop = (exit_on_index ? (it >= Lmin) : (it + 1 >= Lmin)) && (it + 1 < L);
    stream_fwd_rows_kernel<<<w.nchunk, NT, 0, st>>>(C, B, kscale, ahat, w.v_cur, w.u_cur, u_hist + (long long)(it + 1) * B,
                                                    w.part_a, w.part_b, w.state, may_stop ? 1 : 0);
    KCCOT_LAUNCH_CHECK();
    stream_fwd_combine_kernel<<<cgrid, NT, 0, st>>>(w.part_a, w.part_b, w.nchunk, B, ahat, w.v_cur,
                                                    v_hist + (long long)(it + 1) * B, w.state);
    KCCOT_LAUNCH_CHECK();
    if (may_stop) {
      stream_stop_kernel<<<1, 1, 0, st>>>(w.state, it + 1, thresh, kscale, 1);
      KCCOT_LAUNCH_CHECK();
    }
  }
  stream_cost_kernel<<<min(2 * num_sms(), (B + 7) / 8), NT, 0, st>>>(C, B, kscale, w.u_cur, w.v_cur, w.state);
  KCCOT_LAUNCH_CHECK();
  stream_cost_finish_kernel<<<1, 1, 0, st>>>(w.state, kscale, L, cost, nits);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}

int stream_sinkhorn_bwd(const float* C, int B, float eps, int L, const float* u_hist, const float* v_hist,
                        const int32_t* nits, const float* gcost, float* Cbar, void* ws, cudaStream_t st) {
  StreamWs w = carve(ws, B);
  const float kscale = kLog2e / eps, ahat = -log2f((float)B);
  // the saved potentials contain the forward's shift (the global minimum): recompute the same value
  stream_state_init_kernel<<<1, 1, 0, st>>>(w.state);
  KCCOT_LAUNCH_CHECK();
  stream_min_kernel<<<min(4 * num_sms(), (int)(((long long)B * B + NT - 1) / NT)), NT, 0, st>>>(C, (long long)B * B, w.state);
  KCCOT_LAUNCH_CHECK();
  const float* shift_p = &w.state->shift;
  const int cgrid = (B + NT - 1) / NT;
  stream_bwd_seed_kernel<<<w.nchunk, NT, 0, st>>>(C, B, kscale, 1.f / eps, u_hist, v_hist, nits, gcost, shift_p,
                                                  Cbar, w.ubar, w.part_a);
  KCCOT_LAUNCH_CHECK();
  stream_bwd_combine_kernel<<<cgrid, NT, 0, st>>>(w.part_a, w.nchunk, B, 1.f, w.vbar, nullptr, 0);
  KCCOT_LAUNCH_CHECK();
  for (int k = L; k >= 1; --k) {
    stream_bwd_rows_kernel<<<w.nchunk, NT, 0, st>>>(C, B, kscale, ahat, u_hist, v_hist, nits, k, shift_p, w.vbar,
                                                    w.ubar, Cbar, w.part_a);
    KCCOT_LAUNCH_CHECK();
    stream_bwd_combine_kernel<<<cgrid, NT, 0, st>>>(w.part_a, w.nchunk, B, -1.f, w.vbar, nits, k);
    KCCOT_LAUNCH_CHECK();
  }
  return KCCOT_OK;
}

}  // namespace kccot
