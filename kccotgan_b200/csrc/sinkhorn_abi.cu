// C-ABI entry points of the Sinkhorn solve (see include/kccot.h).
#include "sinkhorn.cuh"

using namespace kccot;

namespace {
constexpr int kPersistChunk = 6;     // problems per cooperative launch (their CTAs share the grid)
}

extern "C" {

size_t kccot_sinkhorn_workspace_bytes(int nsolve, int B, int L) {
  (void)L;
  if (B <= kSmallSinkhornMaxB) return align_up(256 + (size_t)(nsolve > 0 ? nsolve : 1) * sizeof(int32_t), 256);
  size_t a = stream_workspace_bytes(B);
  if (persist_supported(B, B, L)) {
    const size_t b = persist_workspace_bytes(nsolve < kPersistChunk ? (nsolve > 0 ? nsolve : 1) : kPersistChunk, B, B, L);
    a = a > b ? a : b;
  }
  return a;
}

int kccot_sinkhorn_fwd(const float* C, int nsolve, int B, float eps, int L, int Lmin, float thresh, int exit_on_index,
                       float* u_hist, float* v_hist, int32_t* nits, float* cost, void* ws, size_t ws_bytes,
                       void* stream) {
  KCCOT_CHECK_ARG(C && u_hist && v_hist && nits && cost, "null pointer");
  KCCOT_CHECK_ARG(nsolve >= 1 && B >= 1 && L >= 0 && eps > 0.f, "bad sizes: nsolve=%d B=%d L=%d eps=%g", nsolve, B, L,
                  (double)eps);
  cudaStream_t st = (cudaStream_t)stream;
  if (B <= kSmallSinkhornMaxB)
    return launch_sinkhorn_fwd_small(C, nsolve, B, eps, L, Lmin, thresh, exit_on_index, u_hist, v_hist, nits, cost, st);
  if (persist_supported(B, B, L) && L >= 1) {
    const long long hs = (long long)(L + 1) * B;
    for (int n0 = 0; n0 < nsolve; n0 += kPersistChunk) {
      const int np = nsolve - n0 < kPersistChunk ? nsolve - n0 : kPersistChunk;
      KCCOT_CHECK_ARG(ws && ws_bytes >= persist_workspace_bytes(np, B, B, L), "workspace too small");
      if (int rc = persist_sinkhorn_fwd(C + (long long)n0 * B * B, np, B, B, 0, eps, L, Lmin, thresh, exit_on_index,
                                        u_hist + n0 * hs, v_hist + n0 * hs, nits + n0, cost + n0, ws, nullptr, nullptr, st))
        return rc;
    }
    return KCCOT_OK;
  }
  KCCOT_CHECK_ARG(ws && ws_bytes >= stream_workspace_bytes(B), "workspace too small");
  for (int n = 0; n < nsolve; ++n) {
    const long long hs = (long long)(L + 1) * B;
    if (int rc = stream_sinkhorn_fwd(C + (long long)n * B * B, B, eps, L, Lmin, thresh, exit_on_index, u_hist + n * hs,
                                     v_hist + n * hs, nits + n, cost + n, ws, st))
      return rc;
  }
  return KCCOT_OK;
}

int kccot_sinkhorn_bwd(const float* C, int nsolve, int B, float eps, int L, const float* u_hist, const float* v_hist,
                       const int32_t* nits, const float* gcost, float* Cbar, void* ws, size_t ws_bytes, void* stream) {
  KCCOT_CHECK_ARG(C && u_hist && v_hist && nits && gcost && Cbar, "null pointer");
  KCCOT_CHECK_ARG(nsolve >= 1 && B >= 1 && L >= 0 && eps > 0.f, "bad sizes");
  cudaStream_t st = (cudaStream_t)stream;
  if (B <= kSmallSinkhornMaxB)
    return launch_sinkhorn_bwd_small(C, nsolve, B, eps, L, u_hist, v_hist, nits, gcost, Cbar, nullptr, st);
  if (persist_supported(B, B, L) && L >= 1) {
    const long long hs = (long long)(L + 1) * B;
    for (int n0 = 0; n0 < nsolve; n0 += kPersistChunk) {
      const int np = nsolve - n0 < kPersistChunk ? nsolve - n0 : kPersistChunk;
      KCCOT_CHECK_ARG(ws && ws_bytes >= persist_workspace_bytes(np, B, B, L), "workspace too small");
      if (int rc = persist_sinkhorn_bwd(C + (long long)n0 * B * B, np, B, B, 0, eps, L, u_hist + n0 * hs, v_hist + n0 * hs,
                                        nits + n0, gcost + n0, 0.f, Cbar + (long long)n0 * B * B, ws, nullptr, nullptr, st))
        return rc;
    }
    return KCCOT_OK;
  }
  KCCOT_CHECK_ARG(ws && ws_bytes >= stream_workspace_bytes(B), "workspace too small");
  for (int n = 0; n < nsolve; ++n) {
    const long long hs = (long long)(L + 1) * B;
    if (int rc = stream_sinkhorn_bwd(C + (long long)n * B * B, B, eps, L, u_hist + n * hs, v_hist + n * hs, nits + n,
                                     gcost + n, Cbar + (long long)n * B * B, ws, st))
      return rc;
  }
  return KCCOT_OK;
}

}  // extern "C"
