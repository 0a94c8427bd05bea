// C-ABI entry points of the row-sharded single problem (BASELINE config 5 on N GPUs; include/kccot.h).
// The kernels exchange the Sinkhorn column sums THEMSELVES through peer-mapped mailboxes (sinkhorn_persist.cu);
// what is left to the caller's communicator (NCCL) are one-off collectives per evaluation: the cost shift (MIN of
// 3 floats), the cost partial sums (SUM of 6 floats), the transposition of the cost adjoints (all-to-all of two
// [Brows, B] panels) and the sum of the two M gradients (SUM of [B, T, J]).
#include "cost.cuh"
#include "sinkhorn.cuh"

using namespace kccot;

namespace {
int fill_comm(ShardComm* c, int nranks, int rank, void* const* mbox_ptrs, void* const* flag_ptrs,
              unsigned long long epoch_base) {
  KCCOT_CHECK_ARG(nranks >= 1 && nranks <= kMaxShardRanks && rank >= 0 && rank < nranks, "bad rank %d of %d (max %d ranks)", rank,
                  nranks, kMaxShardRanks);
  c->nranks = nranks;
  c->rank = rank;
  c->epoch0 = epoch_base;
  for (int r = 0; r < nranks; ++r) {
    KCCOT_CHECK_ARG(nranks == 1 || (mbox_ptrs && flag_ptrs && mbox_ptrs[r] && flag_ptrs[r]), "null mailbox / flag pointer of rank %d", r);
    c->mbox[r] = nranks > 1 ? (float*)mbox_ptrs[r] : nullptr;
    c->flags[r] = nranks > 1 ? (unsigned long long*)flag_ptrs[r] : nullptr;
  }
  return KCCOT_OK;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

__global__ void __launch_bounds__(256) shard_min_kernel(const float* __restrict__ C, long long n, float* __restrict__ out) {
  __shared__ float red[8];
  const float* Cp = C + (long long)blockIdx.x * n;
  float m = 3.0e38f;
  for (long long i = threadIdx.x; i < n; i += 256) m = fminf(m, Cp[i]);
  m = warp_min(m);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) m = fminf(m, red[w]);
    out[blockIdx.x] = fminf(m, red[0]);
  }
}
}  // namespace

extern "C" {

size_t kccot_shard_cost_workspace_bytes(int B, long long K, int Brows) {
  if (B < 1 || K < 1 || Brows < 1) return 0;
  return large_shard_ws_bytes(B, K, Brows);
}

int kccot_shard_cost_fwd(const float* real, const float* fake, int B, long long K, int row0, int Brows, const float* h_fake,
                         const float* m_real, const float* h_real, const float* m_fake, int T, int J, float s,
                         float* C3rows, void* ws, size_t ws_bytes, void* stream) {
  KCCOT_CHECK_ARG(real && fake && h_fake && m_real && h_real && m_fake && C3rows && ws, "null pointer");
  KCCOT_CHECK_ARG(B >= 1 && K >= 1 && T >= 2 && J >= 1, "bad sizes");
  return large_shard_cost_fwd(real, fake, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s, C3rows, ws, ws_bytes,
                              (cudaStream_t)stream);
}

int kccot_shard_cost_bwd(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B, long long K, int row0,
                         int Brows, const float* h_fake, const float* m_real, const float* h_real, const float* m_fake,
                         int T, int J, float s, float* g_fake_rows, float* gh_fake_rows, float* gm_real_part,
                         float* gh_real_rows, float* gm_fake_part, void* ws, size_t ws_bytes, void* stream) {
  KCCOT_CHECK_ARG(Cbar3rows && XYcol && YYcol && h_fake && m_real && h_real && m_fake && ws, "null pointer");
  return large_shard_cost_bwd(Cbar3rows, XYcol, YYcol, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s, g_fake_rows,
                              gh_fake_rows, gm_real_part, gh_real_rows, gm_fake_part, ws, ws_bytes, (cudaStream_t)stream);
}

int kccot_shard_cost_fwd_bf16(const uint16_t* real, const uint16_t* fake, int B, long long K, int row0, int Brows,
                              const float* h_fake, const float* m_real, const float* h_real, const float* m_fake, int T,
                              int J, float s, float* C3rows, void* ws, size_t ws_bytes, void* stream) {
  KCCOT_CHECK_ARG(real && fake && h_fake && m_real && h_real && m_fake && C3rows && ws, "null pointer");
  KCCOT_CHECK_ARG(B >= 1 && K >= 1 && T >= 2 && J >= 1, "bad sizes");
  KCCOT_CHECK_ARG(row0 >= 0 && Brows >= 1 && row0 + Brows <= B, "bad row range [%d, %d) of %d", row0, row0 + Brows, B);
  KCCOT_CHECK_ARG(aligned16(real) && aligned16(fake), "bf16 videos must be 16-byte aligned");
  return large_shard_cost_fwd(real, fake, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s, C3rows, ws, ws_bytes,
                              (cudaStream_t)stream);
}

int kccot_shard_cost_bwd_bf16(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B, long long K, int row0,
                              int Brows, const float* h_fake, const float* m_real, const float* h_real,
                              const float* m_fake, int T, int J, float s, uint16_t* g_fake_rows, float* gh_fake_rows,
                              float* gm_real_part, float* gh_real_rows, float* gm_fake_part, void* ws, size_t ws_bytes,
                              void* stream) {
  KCCOT_CHECK_ARG(Cbar3rows && XYcol && YYcol && h_fake && m_real && h_real && m_fake && ws, "null pointer");
  KCCOT_CHECK_ARG(B >= 1 && K >= 1 && T >= 2 && J >= 1, "bad sizes");
  KCCOT_CHECK_ARG(row0 >= 0 && Brows >= 1 && row0 + Brows <= B, "bad row range [%d, %d) of %d", row0, row0 + Brows, B);
  KCCOT_CHECK_ARG(aligned16(g_fake_rows), "bf16 gradient rows must be 16-byte aligned");
  return large_shard_cost_bwd(Cbar3rows, XYcol, YYcol, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s, g_fake_rows,
                              gh_fake_rows, gm_real_part, gh_real_rows, gm_fake_part, ws, ws_bytes, (cudaStream_t)stream);
}

// ---- shared context frames -----------------------------------------------------------------------------------------
// (ctx_period, ctx_len) with ctx_len == 0 is no hint (the plain entries run); otherwise 0 < ctx_len < ctx_period and
// K % ctx_period == 0.  The column arithmetic of the hinted kernels is 32-bit.
static bool ctx_hint_ok(long long K, long long period, long long len) {
  if (period < 0 || len < 0 || (period == 0 && len != 0)) return false;
  return period == 0 || (len < period && K % period == 0 && K < (1LL << 31) - 64);
}
#define KCCOT_CHECK_CTX(K, period, len) \
  KCCOT_CHECK_ARG(ctx_hint_ok(K, period, len), "bad shared-context hint: period=%lld len=%lld K=%lld", period, len, K)

size_t kccot_shard_cost_workspace_bytes_ctx(int B, long long K, int Brows, long long ctx_period, long long ctx_len) {
  if (B < 1 || K < 1 || Brows < 1 || !ctx_hint_ok(K, ctx_period, ctx_len)) return 0;
  return ctx_len == 0 ? large_shard_ws_bytes(B, K, Brows) : large_shard_ws_bytes_ctx(B, K, Brows, ctx_period, ctx_len);
}

int kccot_shard_cost_fwd_ctx(const float* real, const float* fake, int B, long long K, int row0, int Brows,
                             const float* h_fake, const float* m_real, const float* h_real, const float* m_fake, int T,
                             int J, float s, float* C3rows, void* ws, size_t ws_bytes, void* stream,
                             long long ctx_period, long long ctx_len) {
  KCCOT_CHECK_ARG(real && fake && h_fake && m_real && h_real && m_fake && C3rows && ws, "null pointer");
  KCCOT_CHECK_ARG(B >= 1 && K >= 1 && T >= 2 && J >= 1, "bad sizes");
  KCCOT_CHECK_ARG(row0 >= 0 && Brows >= 1 && row0 + Brows <= B, "bad row range [%d, %d) of %d", row0, row0 + Brows, B);
  KCCOT_CHECK_CTX(K, ctx_period, ctx_len);
  if (ctx_len == 0)
    return kccot_shard_cost_fwd(real, fake, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s, C3rows, ws,
                                ws_bytes, stream);
  return large_shard_cost_fwd_ctx(real, fake, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s, C3rows, ws,
                                  ws_bytes, ctx_period, ctx_len, (cudaStream_t)stream);
}

int kccot_shard_cost_bwd_ctx(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B, long long K, int row0,
                             int Brows, const float* h_fake, const float* m_real, const float* h_real,
                             const float* m_fake, int T, int J, float s, float* g_fake_rows, float* gh_fake_rows,
                             float* gm_real_part, float* gh_real_rows, float* gm_fake_part, void* ws, size_t ws_bytes,
                             void* stream, long long ctx_period, long long ctx_len) {
  KCCOT_CHECK_ARG(Cbar3rows && XYcol && YYcol && h_fake && m_real && h_real && m_fake && ws, "null pointer");
  KCCOT_CHECK_ARG(B >= 1 && K >= 1 && T >= 2 && J >= 1, "bad sizes");
  KCCOT_CHECK_ARG(row0 >= 0 && Brows >= 1 && row0 + Brows <= B, "bad row range [%d, %d) of %d", row0, row0 + Brows, B);
  KCCOT_CHECK_CTX(K, ctx_period, ctx_len);
  if (ctx_len == 0)
    return kccot_shard_cost_bwd(Cbar3rows, XYcol, YYcol, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s,
                                g_fake_rows, gh_fake_rows, gm_real_part, gh_real_rows, gm_fake_part, ws, ws_bytes, stream);
  return large_shard_cost_bwd_ctx(Cbar3rows, XYcol, YYcol, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s,
                                  g_fake_rows, gh_fake_rows, gm_real_part, gh_real_rows, gm_fake_part, ws, ws_bytes,
                                  ctx_period, ctx_len, (cudaStream_t)stream);
}

int kccot_shard_cost_fwd_bf16_ctx(const uint16_t* real, const uint16_t* fake, int B, long long K, int row0, int Brows,
                                  const float* h_fake, const float* m_real, const float* h_real, const float* m_fake,
                                  int T, int J, float s, float* C3rows, void* ws, size_t ws_bytes, void* stream,
                                  long long ctx_period, long long ctx_len) {
  KCCOT_CHECK_ARG(real && fake && h_fake && m_real && h_real && m_fake && C3rows && ws, "null pointer");
  KCCOT_CHECK_ARG(B >= 1 && K >= 1 && T >= 2 && J >= 1, "bad sizes");
  KCCOT_CHECK_ARG(row0 >= 0 && Brows >= 1 && row0 + Brows <= B, "bad row range [%d, %d) of %d", row0, row0 + Brows, B);
  KCCOT_CHECK_ARG(aligned16(real) && aligned16(fake), "bf16 videos must be 16-byte aligned");
  KCCOT_CHECK_CTX(K, ctx_period, ctx_len);
  if (ctx_len == 0)
    return kccot_shard_cost_fwd_bf16(real, fake, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s, C3rows, ws,
                                     ws_bytes, stream);
  return large_shard_cost_fwd_ctx(real, fake, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s, C3rows, ws,
                                  ws_bytes, ctx_period, ctx_len, (cudaStream_t)stream);
}

int kccot_shard_cost_bwd_bf16_ctx(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B, long long K,
                                  int row0, int Brows, const float* h_fake, const float* m_real, const float* h_real,
                                  const float* m_fake, int T, int J, float s, uint16_t* g_fake_rows, float* gh_fake_rows,
                                  float* gm_real_part, float* gh_real_rows, float* gm_fake_part, void* ws,
                                  size_t ws_bytes, void* stream, long long ctx_period, long long ctx_len) {
  KCCOT_CHECK_ARG(Cbar3rows && XYcol && YYcol && h_fake && m_real && h_real && m_fake && ws, "null pointer");
  KCCOT_CHECK_ARG(B >= 1 && K >= 1 && T >= 2 && J >= 1, "bad sizes");
  KCCOT_CHECK_ARG(row0 >= 0 && Brows >= 1 && row0 + Brows <= B, "bad row range [%d, %d) of %d", row0, row0 + Brows, B);
  KCCOT_CHECK_ARG(aligned16(g_fake_rows), "bf16 gradient rows must be 16-byte aligned");
  KCCOT_CHECK_CTX(K, ctx_period, ctx_len);
  if (ctx_len == 0)
    return kccot_shard_cost_bwd_bf16(Cbar3rows, XYcol, YYcol, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s,
                                     g_fake_rows, gh_fake_rows, gm_real_part, gh_real_rows, gm_fake_part, ws, ws_bytes,
                                     stream);
  return large_shard_cost_bwd_ctx(Cbar3rows, XYcol, YYcol, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s,
                                  g_fake_rows, gh_fake_rows, gm_real_part, gh_real_rows, gm_fake_part, ws, ws_bytes,
                                  ctx_period, ctx_len, (cudaStream_t)stream);
}

size_t kccot_shard_sinkhorn_workspace_bytes(int np, int Brows, int B, int L) {
  if (np < 1 || Brows < 1 || B < 1 || L < 1 || !persist_supported(Brows, B, L)) return 0;
  return persist_workspace_bytes(np, Brows, B, L);
}
size_t kccot_shard_mailbox_bytes(int np, int nranks, int B) {
  if (np < 1 || nranks < 1 || B < 1) return 0;
  return persist_mailbox_floats(np, nranks, B) * sizeof(float);
}

int kccot_shard_local_min(const float* Crows, int np, int Brows, int B, float* shift_out, void* stream) {
  KCCOT_CHECK_ARG(Crows && shift_out && np >= 1 && Brows >= 1 && B >= 1, "bad arguments");
  shard_min_kernel<<<np, 256, 0, (cudaStream_t)stream>>>(Crows, (long long)Brows * B, shift_out);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}

int kccot_shard_sinkhorn_fwd(const float* Crows, int np, int Brows, int B, int row0, float eps, int L, int Lmin, float thresh,
                             int exit_on_index, float* u_hist, float* v_hist, int32_t* nits, float* cost_partial,
                             const float* shift, int nranks, int rank, void* const* mbox_ptrs, void* const* flag_ptrs,
                             unsigned long long epoch_base, void* ws, size_t ws_bytes, void* stream) {
  KCCOT_CHECK_ARG(Crows && u_hist && v_hist && nits && cost_partial && shift && ws, "null pointer");
  KCCOT_CHECK_ARG(persist_supported(Brows, B, L) && L >= 1, "row-sharded Sinkhorn needs 64 < B <= 8192, B %% 4 == 0, L >= 1 (B=%d L=%d)",
                  B, L);
  KCCOT_CHECK_ARG(ws_bytes >= persist_workspace_bytes(np, Brows, B, L), "workspace too small");
  ShardComm c;
  if (int rc = fill_comm(&c, nranks, rank, mbox_ptrs, flag_ptrs, epoch_base)) return rc;
  return persist_sinkhorn_fwd(Crows, np, Brows, B, row0, eps, L, Lmin, thresh, exit_on_index, u_hist, v_hist, nits, cost_partial,
                              ws, &c, shift, (cudaStream_t)stream);
}

int kccot_shard_sinkhorn_bwd(const float* Crows, int np, int Brows, int B, int row0, float eps, int L, const float* u_hist,
                             const float* v_hist, const int32_t* nits, const float* gcost, float* Cbar_rows,
                             const float* shift, int nranks, int rank, void* const* mbox_ptrs, void* const* flag_ptrs,
                             unsigned long long epoch_base, void* ws, size_t ws_bytes, void* stream) {
  KCCOT_CHECK_ARG(Crows && u_hist && v_hist && nits && gcost && Cbar_rows && shift && ws, "null pointer");
  KCCOT_CHECK_ARG(persist_supported(Brows, B, L) && L >= 1, "row-sharded Sinkhorn needs 64 < B <= 8192, B %% 4 == 0, L >= 1 (B=%d L=%d)",
                  B, L);
  KCCOT_CHECK_ARG(ws_bytes >= persist_workspace_bytes(np, Brows, B, L), "workspace too small");
  ShardComm c;
  if (int rc = fill_comm(&c, nranks, rank, mbox_ptrs, flag_ptrs, epoch_base)) return rc;
  return persist_sinkhorn_bwd(Crows, np, Brows, B, row0, eps, L, u_hist, v_hist, nits, gcost, 0.f, Cbar_rows, ws,
                              &c, shift, (cudaStream_t)stream);
}

}  // extern "C"
