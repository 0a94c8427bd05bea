// Fused entry points of the mixed Sinkhorn loss (gan_utils.py:204-227): one C-ABI call enqueues the
// whole forward (or backward) chain on the caller's stream.
#include "cost.cuh"
#include "sinkhorn.cuh"

namespace kccot {
namespace {
struct SavedLayout {
  size_t off_C3, off_uh, off_vh, off_nits, off_cost, off_cnt, total;
};
SavedLayout saved_layout(int nprob, int B, int L) {
  SavedLayout s;
  size_t o = 0;
  s.off_C3 = o; o += align_up((size_t)nprob * 3 * B * B * 4, 256);
  s.off_uh = o; o += align_up((size_t)nprob * 3 * (L + 1) * B * 4, 256);
  s.off_vh = o; o += align_up((size_t)nprob * 3 * (L + 1) * B * 4, 256);
  s.off_nits = o; o += align_up((size_t)nprob * 3 * 4, 256);
  s.off_cost = o; o += align_up((size_t)nprob * 3 * 4, 256);
  s.off_cnt = o; o += align_up((size_t)nprob * 4, 256);     // triple-completion counters (SinkhornMix)
  s.total = o;
  return s;
}

__global__ void combine_loss_kernel(const float* __restrict__ cost, int nprob, float* __restrict__ loss,
                                    float* __restrict__ terms) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nprob) return;
  const float xy = cost[3 * p], xx = cost[3 * p + 1], yy = cost[3 * p + 2];
  loss[p] = 2.f * xy - xx - yy;                 // gan_utils.py:225
  if (terms) { terms[3 * p] = xy; terms[3 * p + 1] = xx; terms[3 * p + 2] = yy; }
}

// zeroes the context columns of g [rows][period] (rows = nprob * B * K / period); len % 4 == 0 or scalar stores
__global__ void __launch_bounds__(256) zero_ctx_columns_kernel(float* __restrict__ g, long long rows, long long period,
                                                               long long len) {
  if ((len & 3) == 0 && (period & 3) == 0) {
    const long long per_row = len >> 2, total = rows * per_row;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
      const long long r = i / per_row, c = i - r * per_row;
      reinterpret_cast<float4*>(g + r * period)[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  } else {
    const long long total = rows * len;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
      const long long r = i / len, c = i - r * len;
      g[r * period + c] = 0.f;
    }
  }
}
// bf16 form of zero_ctx_columns_kernel: g [rows][period] of raw bf16 bits
__global__ void __launch_bounds__(256) zero_ctx_columns_bf16_kernel(uint16_t* __restrict__ g, long long rows,
                                                                    long long period, long long len) {
  const long long total = rows * len;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / len, c = i - r * len;
    g[r * period + c] = 0;
  }
}
// bf16 (raw bits) -> fp32, exact; 16-byte aligned src and dst
__global__ void __launch_bounds__(256) widen_bf16_kernel(const uint16_t* __restrict__ src, float* __restrict__ dst,
                                                         long long n) {
  const long long n8 = n >> 3, stride = (long long)gridDim.x * blockDim.x;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += stride) {
    const uint4 v = reinterpret_cast<const uint4*>(src)[i];
    float4* d = reinterpret_cast<float4*>(dst) + 2 * i;
    d[0] = widen_bf16x4(make_uint2(v.x, v.y));
    d[1] = widen_bf16x4(make_uint2(v.z, v.w));
  }
  for (long long i = 8 * n8 + blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += stride)
    dst[i] = __uint_as_float((uint32_t)src[i] << 16);
}
// fp32 -> bf16 (raw bits), round to nearest even; 16-byte aligned src and dst
__global__ void __launch_bounds__(256) narrow_bf16_kernel(const float* __restrict__ src, uint16_t* __restrict__ dst,
                                                          long long n) {
  const long long n8 = n >> 3, stride = (long long)gridDim.x * blockDim.x;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += stride) {
    const float4 a = reinterpret_cast<const float4*>(src)[2 * i], b = reinterpret_cast<const float4*>(src)[2 * i + 1];
    uint4 v;
    v.x = pack_bf16x2(a.x, a.y); v.y = pack_bf16x2(a.z, a.w); v.z = pack_bf16x2(b.x, b.y); v.w = pack_bf16x2(b.z, b.w);
    reinterpret_cast<uint4*>(dst)[i] = v;
  }
  for (long long i = 8 * n8 + blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += stride) {
    const __nv_bfloat16 h = __float2bfloat16_rn(src[i]);
    dst[i] = *reinterpret_cast<const uint16_t*>(&h);
  }
}
int launch_widen(const uint16_t* src, float* dst, long long n, cudaStream_t st) {
  const long long blocks = (n / 8 + 255) / 256;
  widen_bf16_kernel<<<(int)(blocks < 148 * 8 ? (blocks > 0 ? blocks : 1) : 148 * 8), 256, 0, st>>>(src, dst, n);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}
int launch_narrow(const float* src, uint16_t* dst, long long n, cudaStream_t st) {
  const long long blocks = (n / 8 + 255) / 256;
  narrow_bf16_kernel<<<(int)(blocks < 148 * 8 ? (blocks > 0 ? blocks : 1) : 148 * 8), 256, 0, st>>>(src, dst, n);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}

__global__ void expand_gloss_kernel(const float* __restrict__ gloss, int nprob, float* __restrict__ gcost) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nprob) return;
  const float g = gloss[p];
  gcost[3 * p] = 2.f * g; gcost[3 * p + 1] = -g; gcost[3 * p + 2] = -g;
}
}  // namespace
}  // namespace kccot

using namespace kccot;

extern "C" {

size_t kccot_mixed_loss_saved_bytes(int nprob, int B, int L) {
  if (nprob < 1 || B < 1 || L < 0) return 0;
  return saved_layout(nprob, B, L).total;
}

size_t kccot_mixed_loss_workspace_bytes(int nprob, int B, long long K, int L) {
  if (nprob < 1 || B < 1 || K < 1) return 0;
  size_t a = kccot_mixed_cost_workspace_bytes(nprob, B, K);
  size_t b = kccot_sinkhorn_workspace_bytes(3 * nprob, B, L);
  // backward: Cbar3 + gcost + the larger of (Sinkhorn workspace, W' scratch)
  size_t c = align_up((size_t)nprob * 3 * B * B * 4, 256) + align_up((size_t)nprob * 3 * 4, 256) +
             (b > kccot_mixed_cost_bwd_workspace_bytes(nprob, B, K) ? b : kccot_mixed_cost_bwd_workspace_bytes(nprob, B, K));
  size_t m = a > b ? a : b;
  return align_up(m > c ? m : c, 256);
}

}  // extern "C"

namespace kccot {
// bf16 videos: the native path (bf16 tensor-core kernels, results bit-identical to the fp32 call on the widened
// videos) is chosen from the shape and the path flag alone, so that the workspace query knows it
static bool bf16_native(int B, long long K, int flags) {
  return (flags & 3) != KCCOT_PATH_SIMT && B <= 64 && B % 8 == 0 && K % 8 == 0 && K >= 128;
}
// one fp32 copy of a video in the widened path's workspace
static size_t widened_bytes(int nprob, int B, long long K) { return align_up((size_t)nprob * B * K * 4, 256); }
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// real16 / fake16 set: bf16 videos on the native path (real / fake unused)
static int loss_fwd(const float* real, const float* fake, const uint16_t* real16, const uint16_t* fake16, int nprob,
                    int B, long long K, const float* h_fake, const float* m_real, const float* h_real,
                    const float* m_fake, int T, int J, float s, float eps, int L, void* saved, float* loss,
                    float* terms, void* ws, size_t ws_bytes, int flags, void* stream) {
  KCCOT_CHECK_ARG(saved && loss && ws, "null pointer");
  KCCOT_CHECK_ARG(L >= 0 && eps > 0.f, "bad eps / L");
  const SavedLayout sl = saved_layout(nprob, B, L);
  char* sv = (char*)saved;
  float* C3 = (float*)(sv + sl.off_C3);
  const bool small = B <= kSmallSinkhornMaxB;      // loss combination folded into the Sinkhorn kernel
  int* counters = (int*)(sv + sl.off_cnt);
  if (int rc = real16 ? mixed_cost_fwd_bf16_tc(real16, fake16, nprob, B, K, h_fake, m_real, h_real, m_fake, T, J, s,
                                               C3, ws, ws_bytes, (cudaStream_t)stream, small ? counters : nullptr)
                      : mixed_cost_fwd_impl(real, fake, nprob, B, K, h_fake, m_real, h_real, m_fake, T, J, s, C3, ws,
                                            ws_bytes, flags, stream, small ? counters : nullptr))
    return rc;
  // Lmin = 100, thresh = 1e-2, break on the iteration COUNT: compute_sinkhorn, gan_utils.py:144-160
  if (small) {
    SinkhornMix mix;
    mix.loss = loss; mix.terms = terms; mix.counter = counters;
    KCCOT_CHECK_ARG(L >= 0 && eps > 0.f, "bad eps / L");
    return launch_sinkhorn_fwd_small(C3, 3 * nprob, B, eps, L, 100, 1e-2f, 0, (float*)(sv + sl.off_uh),
                                     (float*)(sv + sl.off_vh), (int32_t*)(sv + sl.off_nits), (float*)(sv + sl.off_cost),
                                     (cudaStream_t)stream, mix);
  }
  if (int rc = kccot_sinkhorn_fwd(C3, 3 * nprob, B, eps, L, 100, 1e-2f, 0, (float*)(sv + sl.off_uh),
                                  (float*)(sv + sl.off_vh), (int32_t*)(sv + sl.off_nits), (float*)(sv + sl.off_cost), ws,
                                  ws_bytes, stream))
    return rc;
  combine_loss_kernel<<<(nprob + 127) / 128, 128, 0, (cudaStream_t)stream>>>((const float*)(sv + sl.off_cost), nprob, loss,
                                                                           terms);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}

// reverse Sinkhorn solves: Cbar3 (the 2, -1, -1 weights applied) at the start of `ws`; *ws2 = the rest of it
static int loss_bwd_cbar(const float* gloss, int nprob, int B, float eps, int L, const void* saved, void* ws,
                         size_t ws_bytes, void* stream, float** Cbar3_out, void** ws2_out, size_t* ws2_bytes_out) {
  KCCOT_CHECK_ARG(gloss && saved && ws, "null pointer");
  const SavedLayout sl = saved_layout(nprob, B, L);
  const char* sv = (const char*)saved;
  const size_t cb_bytes = align_up((size_t)nprob * 3 * B * B * 4, 256);
  const size_t gc_bytes = align_up((size_t)nprob * 3 * 4, 256);
  KCCOT_CHECK_ARG(ws_bytes >= cb_bytes + gc_bytes + 256, "workspace too small");
  float* Cbar3 = (float*)ws;
  float* gcost = (float*)((char*)ws + cb_bytes);
  void* ws2 = (char*)ws + cb_bytes + gc_bytes;
  const size_t ws2_bytes = ws_bytes - cb_bytes - gc_bytes;
  if (B <= kSmallSinkhornMaxB) {                   // the 2, -1, -1 weights are applied inside the kernel
    SinkhornMix mix;
    mix.gloss = gloss;
    if (int rc = launch_sinkhorn_bwd_small((const float*)(sv + sl.off_C3), 3 * nprob, B, eps, L,
                                           (const float*)(sv + sl.off_uh), (const float*)(sv + sl.off_vh),
                                           (const int32_t*)(sv + sl.off_nits), nullptr, Cbar3, nullptr,
                                           (cudaStream_t)stream, mix))
      return rc;
  } else {
    expand_gloss_kernel<<<(nprob + 127) / 128, 128, 0, (cudaStream_t)stream>>>(gloss, nprob, gcost);
    KCCOT_LAUNCH_CHECK();
    if (int rc = kccot_sinkhorn_bwd((const float*)(sv + sl.off_C3), 3 * nprob, B, eps, L, (const float*)(sv + sl.off_uh),
                                    (const float*)(sv + sl.off_vh), (const int32_t*)(sv + sl.off_nits), gcost, Cbar3, ws2,
                                    ws2_bytes, stream))
      return rc;
  }
  *Cbar3_out = Cbar3;
  *ws2_out = ws2;
  *ws2_bytes_out = ws2_bytes;
  return KCCOT_OK;
}

// g_fake's context columns: skipped by the tensor-core path, filled with the plain gradient by the others — zero
// either way (left alone by an accumulating call)
static int zero_ctx_columns(void* g_fake, bool bf16, int nprob, int B, long long K, int flags, long long ctx_period,
                            long long ctx_len, cudaStream_t st) {
  if (g_fake && ctx_len > 0 && K % ctx_period == 0 && !(flags & KCCOT_FLAG_ACCUMULATE)) {
    const long long rows = (long long)nprob * B * (K / ctx_period);
    const long long work = bf16 ? rows * ctx_len : rows * ((ctx_len + 3) / 4);
    const int grid = (int)((work + 255) / 256 < 148 * 8 ? (work + 255) / 256 : 148 * 8);
    if (bf16)
      zero_ctx_columns_bf16_kernel<<<grid, 256, 0, st>>>((uint16_t*)g_fake, rows, ctx_period, ctx_len);
    else
      zero_ctx_columns_kernel<<<grid, 256, 0, st>>>((float*)g_fake, rows, ctx_period, ctx_len);
    KCCOT_LAUNCH_CHECK();
  }
  return KCCOT_OK;
}
}  // namespace kccot

extern "C" {

int kccot_mixed_loss_fwd(const float* real, const float* fake, int nprob, int B, long long K, const float* h_fake,
                         const float* m_real, const float* h_real, const float* m_fake, int T, int J, float s, float eps,
                         int L, void* saved, float* loss, float* terms, void* ws, size_t ws_bytes, int flags,
                         void* stream) {
  return loss_fwd(real, fake, nullptr, nullptr, nprob, B, K, h_fake, m_real, h_real, m_fake, T, J, s, eps, L, saved,
                  loss, terms, ws, ws_bytes, flags, stream);
}

int kccot_mixed_loss_bwd(const float* gloss, const float* real, const float* fake, int nprob, int B, long long K,
                         const float* h_fake, const float* m_real, const float* h_real, const float* m_fake, int T,
                         int J, float s, float eps, int L, const void* saved, float* g_real, float* g_fake,
                         float* gh_fake, float* gm_real, float* gh_real, float* gm_fake, void* ws, size_t ws_bytes,
                         int flags, void* stream) {
  float* Cbar3;
  void* ws2;
  size_t ws2_bytes;
  if (int rc = loss_bwd_cbar(gloss, nprob, B, eps, L, saved, ws, ws_bytes, stream, &Cbar3, &ws2, &ws2_bytes)) return rc;
  return kccot_mixed_cost_bwd(Cbar3, real, fake, nprob, B, K, h_fake, m_real, h_real, m_fake, T, J, s, g_real, g_fake,
                              gh_fake, gm_real, gh_real, gm_fake, ws2, ws2_bytes, flags, stream);
}


int kccot_mixed_loss_fwd_ctx(const float* real, const float* fake, int nprob, int B, long long K, const float* h_fake,
                             const float* m_real, const float* h_real, const float* m_fake, int T, int J, float s,
                             float eps, int L, void* saved, float* loss, float* terms, void* ws, size_t ws_bytes,
                             int flags, void* stream, long long ctx_period, long long ctx_len) {
  KCCOT_CHECK_ARG(ctx_period >= 0 && ctx_len >= 0 && (ctx_len == 0 || ctx_len < ctx_period),
                  "bad shared-context hint: period=%lld len=%lld", ctx_period, ctx_len);
  CtxScope scope(ctx_period, ctx_len);
  return kccot_mixed_loss_fwd(real, fake, nprob, B, K, h_fake, m_real, h_real, m_fake, T, J, s, eps, L, saved, loss,
                              terms, ws, ws_bytes, flags, stream);
}

int kccot_mixed_loss_bwd_ctx(const float* gloss, const float* real, const float* fake, int nprob, int B, long long K,
                             const float* h_fake, const float* m_real, const float* h_real, const float* m_fake, int T,
                             int J, float s, float eps, int L, const void* saved, float* g_real, float* g_fake,
                             float* gh_fake, float* gm_real, float* gh_real, float* gm_fake, void* ws, size_t ws_bytes,
                             int flags, void* stream, long long ctx_period, long long ctx_len) {
  KCCOT_CHECK_ARG(ctx_period >= 0 && ctx_len >= 0 && (ctx_len == 0 || ctx_len < ctx_period),
                  "bad shared-context hint: period=%lld len=%lld", ctx_period, ctx_len);
  CtxScope scope(ctx_period, ctx_len);
  if (int rc = kccot_mixed_loss_bwd(gloss, real, fake, nprob, B, K, h_fake, m_real, h_real, m_fake, T, J, s, eps, L, saved,
                                    g_real, g_fake, gh_fake, gm_real, gh_real, gm_fake, ws, ws_bytes, flags, stream))
    return rc;
  return zero_ctx_columns(g_fake, false, nprob, B, K, flags, ctx_period, ctx_len, (cudaStream_t)stream);
}

size_t kccot_mixed_loss_workspace_bytes_bf16(int nprob, int B, long long K, int L, int flags) {
  const size_t base = kccot_mixed_loss_workspace_bytes(nprob, B, K, L);
  if (!base || bf16_native(B, K, flags)) return base;
  return 4 * widened_bytes(nprob, B, K) + base;       // widened real, fake | fp32 gradient scratch | fp32 workspace
}

int kccot_mixed_loss_fwd_bf16(const uint16_t* real, const uint16_t* fake, int nprob, int B, long long K,
                              const float* h_fake, const float* m_real, const float* h_real, const float* m_fake, int T,
                              int J, float s, float eps, int L, void* saved, float* loss, float* terms, void* ws,
                              size_t ws_bytes, int flags, void* stream, long long ctx_period, long long ctx_len) {
  KCCOT_CHECK_ARG(!(flags & KCCOT_FLAG_ACCUMULATE), "KCCOT_FLAG_ACCUMULATE is not supported with bf16 videos");
  KCCOT_CHECK_ARG(real && fake, "null pointer");
  KCCOT_CHECK_ARG(aligned16(real) && aligned16(fake), "bf16 videos must be 16-byte aligned");
  KCCOT_CHECK_ARG(nprob >= 1 && B >= 1 && K >= 1, "bad sizes: nprob=%d B=%d K=%lld", nprob, B, K);
  KCCOT_CHECK_ARG(ctx_period >= 0 && ctx_len >= 0 && (ctx_len == 0 || ctx_len < ctx_period),
                  "bad shared-context hint: period=%lld len=%lld", ctx_period, ctx_len);
  CtxScope scope(ctx_period, ctx_len);
  if (bf16_native(B, K, flags))
    return loss_fwd(nullptr, nullptr, real, fake, nprob, B, K, h_fake, m_real, h_real, m_fake, T, J, s, eps, L, saved,
                    loss, terms, ws, ws_bytes, flags, stream);
  // widened path: fp32 copies in the workspace, then the fp32 chain on them
  const size_t vb = widened_bytes(nprob, B, K);
  KCCOT_CHECK_ARG(ws && ws_bytes >= 4 * vb + 256, "workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const long long n = (long long)nprob * B * K;
  float* R32 = (float*)ws;
  float* F32 = (float*)((char*)ws + vb);
  if (int rc = launch_widen(real, R32, n, st)) return rc;
  if (int rc = launch_widen(fake, F32, n, st)) return rc;
  return loss_fwd(R32, F32, nullptr, nullptr, nprob, B, K, h_fake, m_real, h_real, m_fake, T, J, s, eps, L, saved, loss,
                  terms, (char*)ws + 4 * vb, ws_bytes - 4 * vb, flags, stream);
}

int kccot_mixed_loss_bwd_bf16(const float* gloss, const uint16_t* real, const uint16_t* fake, int nprob, int B,
                              long long K, const float* h_fake, const float* m_real, const float* h_real,
                              const float* m_fake, int T, int J, float s, float eps, int L, const void* saved,
                              uint16_t* g_real, uint16_t* g_fake, float* gh_fake, float* gm_real, float* gh_real,
                              float* gm_fake, void* ws, size_t ws_bytes, int flags, void* stream, long long ctx_period,
                              long long ctx_len) {
  KCCOT_CHECK_ARG(!(flags & KCCOT_FLAG_ACCUMULATE), "KCCOT_FLAG_ACCUMULATE is not supported with bf16 videos");
  KCCOT_CHECK_ARG(real && fake, "null pointer");
  KCCOT_CHECK_ARG(aligned16(real) && aligned16(fake) && aligned16(g_real) && aligned16(g_fake),
                  "bf16 videos and their gradients must be 16-byte aligned");
  KCCOT_CHECK_ARG(nprob >= 1 && B >= 1 && K >= 1, "bad sizes: nprob=%d B=%d K=%lld", nprob, B, K);
  KCCOT_CHECK_ARG(ctx_period >= 0 && ctx_len >= 0 && (ctx_len == 0 || ctx_len < ctx_period),
                  "bad shared-context hint: period=%lld len=%lld", ctx_period, ctx_len);
  cudaStream_t st = (cudaStream_t)stream;
  if (bf16_native(B, K, flags)) {
    CtxScope scope(ctx_period, ctx_len);
    float* Cbar3;
    void* ws2;
    size_t ws2_bytes;
    if (int rc = loss_bwd_cbar(gloss, nprob, B, eps, L, saved, ws, ws_bytes, stream, &Cbar3, &ws2, &ws2_bytes)) return rc;
    if (int rc = mixed_cost_bwd_bf16_tc(Cbar3, real, fake, nprob, B, K, h_fake, m_real, h_real, m_fake, T, J, s, g_real,
                                        g_fake, gh_fake, gm_real, gh_real, gm_fake, ws2, ws2_bytes, st))
      return rc;
    return zero_ctx_columns(g_fake, true, nprob, B, K, flags, ctx_period, ctx_len, st);
  }
  // widened path: the fp32 backward on fp32 copies into fp32 scratch, rounded to bf16 at the end
  const size_t vb = widened_bytes(nprob, B, K);
  KCCOT_CHECK_ARG(ws && ws_bytes >= 4 * vb + 256, "workspace too small");
  const long long n = (long long)nprob * B * K;
  char* w = (char*)ws;
  float* R32 = (float*)w;
  float* F32 = (float*)(w + vb);
  float* GR32 = g_real ? (float*)(w + 2 * vb) : nullptr;
  float* GF32 = g_fake ? (float*)(w + 3 * vb) : nullptr;
  if (int rc = launch_widen(real, R32, n, st)) return rc;
  if (int rc = launch_widen(fake, F32, n, st)) return rc;
  if (int rc = kccot_mixed_loss_bwd_ctx(gloss, R32, F32, nprob, B, K, h_fake, m_real, h_real, m_fake, T, J, s, eps, L,
                                        saved, GR32, GF32, gh_fake, gm_real, gh_real, gm_fake, w + 4 * vb,
                                        ws_bytes - 4 * vb, flags, stream, ctx_period, ctx_len))
    return rc;
  if (g_real)
    if (int rc = launch_narrow(GR32, g_real, n, st)) return rc;
  if (g_fake)
    if (int rc = launch_narrow(GF32, g_fake, n, st)) return rc;
  return KCCOT_OK;
}

}  // extern "C"
