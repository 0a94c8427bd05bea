// C-ABI entry points of the cost path (see include/kccot.h): kernel-path selection, workspace
// carving, launches.  No allocation, no synchronisation.
#include "cost.cuh"

namespace kccot {
namespace {

constexpr long long kTcTile = 128LL * 128LL;

size_t simt_part_bytes(int nprob, int Bx, int By, long long K) {
  int ks;
  long long slab;
  choose_ksplit_simt(nprob, Bx, By, K, &ks, &slab);
  return (size_t)nprob * ks * Bx * By * sizeof(float);
}
size_t tc_part_bytes(int nprob, int R, long long K) {
  int ks, kbps;
  tc_sqdist_plan(nprob, R, K, &ks, &kbps);
  return (size_t)nprob * ks * kTcTile * sizeof(float);
}
int pick_path(int flags, bool tc_ok) {
  const int want = flags & 3;
  if (want == KCCOT_PATH_SIMT) return KCCOT_PATH_SIMT;
  if (want == KCCOT_PATH_TCGEN05) return tc_ok ? KCCOT_PATH_TCGEN05 : -1;
  return tc_ok ? KCCOT_PATH_TCGEN05 : KCCOT_PATH_SIMT;
}
int check_common(int nprob, int Bx, int By, long long K) {
  KCCOT_CHECK_ARG(nprob >= 1 && Bx >= 1 && By >= 1 && K >= 1, "bad sizes: nprob=%d Bx=%d By=%d K=%lld", nprob, Bx,
                  By, K);
  return KCCOT_OK;
}
// the three blocks (xy, xx, yy — gan_utils.py:221-223) of the mixed cost, without their partials
void mixed_blocks(CostBlocks& blocks, const float* h_fake, const float* m_real, const float* h_real, const float* m_fake,
                  int B, float* C3, int* zero_counters) {
  blocks.zero = zero_counters;
  const long long BB = (long long)B * B;
  const float* hs[3] = {h_fake, h_real, h_fake};
  const float* Ms[3] = {m_real, m_real, m_fake};
  for (int q = 0; q < 3; ++q) {
    CostBlock& b = blocks.b[q];
    b.h1 = hs[q]; b.M1 = Ms[q]; b.h2 = nullptr; b.M2 = nullptr;
    b.C = C3 + q * BB; b.C_prob_stride = 3 * BB; b.Bx = B; b.By = B; b.zero_diag = q > 0;
  }
}
// the partials of the stacked-row tensor-core kernel: blocks of the [2B x 2B] tile
void mixed_blocks_tc(CostBlocks& blocks, const float* part, int B, int ks) {
  const int roff[3] = {0, 0, B}, coff[3] = {B, 0, B};
  for (int q = 0; q < 3; ++q) {
    CostBlock& b = blocks.b[q];
    b.part = part; b.prob_stride = (long long)ks * kTcTile; b.ks_stride = kTcTile; b.ld = 128;
    b.nks = ks; b.row_off = roff[q]; b.col_off = coff[q]; b.sym = 1; b.tiled = 1;
  }
}
// martingale terms of the mixed adjoint: xy = (h_fake, m_real), xx = (h_real, m_real), yy = (h_fake, m_fake)
MartJobs mixed_mart_jobs(const float* Cbar3, int B, const float* h_fake, const float* m_real, const float* h_real,
                         const float* m_fake, float* gh_fake, float* gm_real, float* gh_real, float* gm_fake, int acc) {
  const long long BB = (long long)B * B, cprob = 3 * BB;
  const float* Cxy = Cbar3;
  const float* Cxx = Cbar3 + BB;
  const float* Cyy = Cbar3 + 2 * BB;
  MartJobs jobs{};
  jobs.j[0] = MartJob{gh_fake, Cxy, m_real, Cyy, m_fake, cprob, B, B, B, 0, 0, acc};
  jobs.j[1] = MartJob{gm_real, Cxy, h_fake, Cxx, h_real, cprob, B, B, B, 1, 1, acc};
  jobs.j[2] = MartJob{gh_real, Cxx, m_real, nullptr, nullptr, cprob, B, B, B, 0, 0, acc};
  jobs.j[3] = MartJob{gm_fake, Cyy, h_fake, nullptr, nullptr, cprob, B, B, B, 1, 1, acc};
  return jobs;
}
// The martingale adjoint (a few MFLOP, ~10 us of latency) and the gradient GEMM both depend on Cbar3 only: the
// small kernel goes first on the side stream and the persistent GEMM CTAs (`grad`) fill in around it.
template <typename Grad>
int mart_beside_grad(const MartJobs& jobs, int nprob, int T, int J, float s, cudaStream_t st, Grad grad) {
  SideLane* lane = side_lane();
  cudaStream_t ms = st;
  if (lane) {
    KCCOT_CUDA(cudaEventRecord(lane->fork, st));
    KCCOT_CUDA(cudaStreamWaitEvent(lane->stream, lane->fork, 0));
    ms = lane->stream;
  }
  if (int rc = launch_martingale_jobs(jobs, 4, nprob, T, J, s, ms)) return rc;
  if (lane) KCCOT_CUDA(cudaEventRecord(lane->join, lane->stream));
  if (int rc = grad()) return rc;
  if (lane) KCCOT_CUDA(cudaStreamWaitEvent(st, lane->join, 0));
  return KCCOT_OK;
}

}  // namespace
}  // namespace kccot

using namespace kccot;

extern "C" {

size_t kccot_cost_workspace_bytes(int nprob, int Bx, int By, long long K) {
  if (nprob < 1 || Bx < 1 || By < 1 || K < 1) return 0;
  size_t a = simt_part_bytes(nprob, Bx, By, K);
  // the stacked-row tensor-core kernel takes [x; y] (rows Bx + By) or, for a self-cost (x == y), x alone (rows Bx):
  // size for whichever the launcher may pick
  if (Bx + By <= 128 || (Bx == By && Bx <= 128)) {
    const size_t t = tc_part_bytes(nprob, Bx + By <= 128 ? Bx + By : Bx, K);
    a = a > t ? a : t;
  }
  if (large_path_wanted(Bx, By, false)) {
    const size_t l = large_cost_fwd_ws_bytes(Bx, By, K, false, false);
    a = a > l ? a : l;
  }
  return align_up(a, 256);
}

int kccot_cost_fwd(const float* x, const float* y, int nprob, int Bx, int By, long long K, const float* h1,
                   const float* M1, const float* h2, const float* M2, int T, int J, float s, float* C, void* ws,
                   size_t ws_bytes, int flags, void* stream) {
  if (int rc = check_common(nprob, Bx, By, K)) return rc;
  KCCOT_CHECK_ARG(x && y && C && ws, "null pointer");
  KCCOT_CHECK_ARG((h1 == nullptr) == (M1 == nullptr) && (h2 == nullptr) == (M2 == nullptr),
                  "h and M must be given in pairs");
  KCCOT_CHECK_ARG(!h1 || (T >= 2 && J >= 1), "martingale term needs T >= 2, J >= 1 (T=%d J=%d)", T, J);
  cudaStream_t st = (cudaStream_t)stream;
  const bool same = (x == y);
  KCCOT_CHECK_ARG(!same || Bx == By, "x == y requires Bx == By");
  if ((flags & 3) != KCCOT_PATH_SIMT && large_path_wanted(Bx, By, same)) {
    for (int p = 0; p < nprob; ++p) {
      const long long hm = (long long)T * J;
      if (int rc = large_cost_fwd(x + (long long)p * Bx * K, same ? x + (long long)p * Bx * K : y + (long long)p * By * K, Bx, By,
                                  K, h1 ? h1 + p * Bx * hm : nullptr, M1 ? M1 + p * By * hm : nullptr,
                                  h2 ? h2 + p * Bx * hm : nullptr, M2 ? M2 + p * By * hm : nullptr, T, J, s,
                                  C + (long long)p * Bx * By, ws, ws_bytes, st))
        return rc;
    }
    return KCCOT_OK;
  }
  const bool tc_ok = same ? tc_sqdist_supported(x, nullptr, Bx, 0, K) : tc_sqdist_supported(x, y, Bx, By, K);
  const int path = pick_path(flags, tc_ok);
  if (path < 0) {
    set_error("tcgen05 path requested but unsupported for Bx=%d By=%d K=%lld (needs rows<=128, B%%8==0, K%%4==0, 16-B aligned)",
              Bx, By, K);
    return KCCOT_EUNSUPPORTED;
  }
  CostBlocks blocks{};
  CostBlock& b = blocks.b[0];
  b.h1 = h1; b.M1 = M1; b.h2 = h2; b.M2 = M2;
  b.C = C; b.C_prob_stride = (long long)Bx * By; b.Bx = Bx; b.By = By; b.zero_diag = same ? 1 : 0;
  b.part = (const float*)ws;
  if (path == KCCOT_PATH_TCGEN05) {
    const int R = same ? Bx : Bx + By;
    int ks, kbps;
    tc_sqdist_plan(nprob, R, K, &ks, &kbps);
    KCCOT_CHECK_ARG(ws_bytes >= (size_t)nprob * ks * kTcTile * 4, "workspace too small");
    if (int rc = launch_sqdist_partials_tc(x, same ? nullptr : y, nprob, Bx, same ? 0 : By, K, ks, kbps, (float*)ws, st))
      return rc;
    b.prob_stride = (long long)ks * kTcTile; b.ks_stride = kTcTile; b.ld = 128; b.nks = ks;
    b.row_off = 0; b.col_off = same ? 0 : Bx; b.sym = 1; b.tiled = 1;
  } else {
    int ks;
    long long slab;
    choose_ksplit_simt(nprob, Bx, By, K, &ks, &slab);
    KCCOT_CHECK_ARG(ws_bytes >= (size_t)nprob * ks * Bx * By * 4, "workspace too small");
    if (int rc = launch_sqdist_partials_simt(x, y, nprob, Bx, By, K, ks, slab, (float*)ws, st)) return rc;
    b.prob_stride = (long long)ks * Bx * By; b.ks_stride = (long long)Bx * By; b.ld = By; b.nks = ks;
    b.row_off = 0; b.col_off = 0;
  }
  return launch_cost_finalize(blocks, 1, nprob, T, J, s, st);
}

size_t kccot_mixed_cost_workspace_bytes(int nprob, int B, long long K) {
  if (nprob < 1 || B < 1 || K < 1) return 0;
  size_t a = 3 * align_up(simt_part_bytes(nprob, B, B, K), 256);
  if (2 * B <= 128) a = a > tc_part_bytes(nprob, 2 * B, K) ? a : tc_part_bytes(nprob, 2 * B, K);
  if (large_path_wanted(B, B, false)) {
    const size_t l = large_cost_fwd_ws_bytes(B, B, K, false, true);
    a = a > l ? a : l;
  }
  return align_up(a, 256);
}

int kccot_mixed_cost_fwd(const float* real, const float* fake, int nprob, int B, long long K, const float* h_fake,
                         const float* m_real, const float* h_real, const float* m_fake, int T, int J, float s,
                         float* C3, void* ws, size_t ws_bytes, int flags, void* stream) {
  return kccot::mixed_cost_fwd_impl(real, fake, nprob, B, K, h_fake, m_real, h_real, m_fake, T, J, s, C3, ws, ws_bytes,
                                    flags, stream, nullptr);
}
}  // extern "C"

namespace kccot {
int mixed_cost_fwd_impl(const float* real, const float* fake, int nprob, int B, long long K, const float* h_fake,
                        const float* m_real, const float* h_real, const float* m_fake, int T, int J, float s,
                        float* C3, void* ws, size_t ws_bytes, int flags, void* stream, int* zero_counters) {
  if (int rc = check_common(nprob, B, B, K)) return rc;
  KCCOT_CHECK_ARG(real && fake && h_fake && m_real && h_real && m_fake && C3 && ws, "null pointer");
  KCCOT_CHECK_ARG(T >= 2 && J >= 1, "martingale term needs T >= 2, J >= 1 (T=%d J=%d)", T, J);
  cudaStream_t st = (cudaStream_t)stream;
  if ((flags & 3) != KCCOT_PATH_SIMT && real != fake && large_path_wanted(B, B, false)) {
    const long long hm = (long long)B * T * J;
    for (int p = 0; p < nprob; ++p)
      if (int rc = large_mixed_cost_fwd(real + (long long)p * B * K, fake + (long long)p * B * K, B, K, h_fake + p * hm,
                                        m_real + p * hm, h_real + p * hm, m_fake + p * hm, T, J, s,
                                        C3 + (long long)p * 3 * B * B, ws, ws_bytes, st))
        return rc;
    if (zero_counters) KCCOT_CUDA(cudaMemsetAsync(zero_counters, 0, (size_t)nprob * sizeof(int), st));
    return KCCOT_OK;
  }
  const bool tc_ok = (real != fake) && tc_sqdist_supported(real, fake, B, B, K);
  const int path = pick_path(flags, tc_ok);
  if (path < 0) {
    set_error("tcgen05 path requested but unsupported for B=%d K=%lld", B, K);
    return KCCOT_EUNSUPPORTED;
  }
  CostBlocks blocks{};
  const long long BB = (long long)B * B;
  mixed_blocks(blocks, h_fake, m_real, h_real, m_fake, B, C3, zero_counters);
  if (path == KCCOT_PATH_TCGEN05) {
    int ks, kbps;
    tc_sqdist_plan(nprob, 2 * B, K, &ks, &kbps);
    KCCOT_CHECK_ARG(ws_bytes >= (size_t)nprob * ks * kTcTile * 4, "workspace too small");
    if (int rc = launch_sqdist_partials_tc(real, fake, nprob, B, B, K, ks, kbps, (float*)ws, st)) return rc;
    mixed_blocks_tc(blocks, (const float*)ws, B, ks);
  } else {
    int ks;
    long long slab;
    choose_ksplit_simt(nprob, B, B, K, &ks, &slab);
    const size_t one = align_up((size_t)nprob * ks * BB * 4, 256);
    KCCOT_CHECK_ARG(ws_bytes >= 3 * one, "workspace too small");
    const float* xs[3] = {real, real, fake};
    const float* ys[3] = {fake, real, fake};
    for (int q = 0; q < 3; ++q) {
      float* part = (float*)((char*)ws + q * one);
      if (int rc = launch_sqdist_partials_simt(xs[q], ys[q], nprob, B, B, K, ks, slab, part, st)) return rc;
      CostBlock& b = blocks.b[q];
      b.part = part; b.prob_stride = (long long)ks * BB; b.ks_stride = BB; b.ld = B; b.nks = ks;
      b.row_off = 0; b.col_off = 0;
    }
  }
  return launch_cost_finalize(blocks, 3, nprob, T, J, s, st);
}

int mixed_cost_fwd_bf16_tc(const uint16_t* real, const uint16_t* fake, int nprob, int B, long long K,
                           const float* h_fake, const float* m_real, const float* h_real, const float* m_fake, int T,
                           int J, float s, float* C3, void* ws, size_t ws_bytes, cudaStream_t st, int* zero_counters) {
  if (int rc = check_common(nprob, B, B, K)) return rc;
  KCCOT_CHECK_ARG(real && fake && h_fake && m_real && h_real && m_fake && C3 && ws, "null pointer");
  KCCOT_CHECK_ARG(T >= 2 && J >= 1, "martingale term needs T >= 2, J >= 1 (T=%d J=%d)", T, J);
  KCCOT_CHECK_ARG(tc_sqdist_bf16_supported(B, B, K), "bf16 tensor-core path unsupported for B=%d K=%lld", B, K);
  CostBlocks blocks{};
  mixed_blocks(blocks, h_fake, m_real, h_real, m_fake, B, C3, zero_counters);
  int ks, kbps;
  tc_sqdist_plan(nprob, 2 * B, K, &ks, &kbps);
  KCCOT_CHECK_ARG(ws_bytes >= (size_t)nprob * ks * kTcTile * 4, "workspace too small");
  if (int rc = launch_sqdist_partials_tc_bf16(real, fake, nprob, B, B, K, ks, kbps, (float*)ws, st)) return rc;
  mixed_blocks_tc(blocks, (const float*)ws, B, ks);
  return launch_cost_finalize(blocks, 3, nprob, T, J, s, st);
}

int mixed_cost_bwd_bf16_tc(const float* Cbar3, const uint16_t* real, const uint16_t* fake, int nprob, int B,
                           long long K, const float* h_fake, const float* m_real, const float* h_real,
                           const float* m_fake, int T, int J, float s, uint16_t* g_real, uint16_t* g_fake,
                           float* gh_fake, float* gm_real, float* gh_real, float* gm_fake, void* ws, size_t ws_bytes,
                           cudaStream_t st) {
  if (int rc = check_common(nprob, B, B, K)) return rc;
  KCCOT_CHECK_ARG(Cbar3 && real && fake && h_fake && m_real && h_real && m_fake, "null pointer");
  KCCOT_CHECK_ARG(ws && ws_bytes >= tc_grad_ws_bytes(nprob), "workspace too small");
  const MartJobs jobs = mixed_mart_jobs(Cbar3, B, h_fake, m_real, h_real, m_fake, gh_fake, gm_real, gh_real, gm_fake, 0);
  return mart_beside_grad(jobs, nprob, T, J, s, st, [&] {
    return launch_grad_tc_bf16(Cbar3, real, fake, nprob, B, K, s, g_real, g_fake, (float*)ws, st);
  });
}
}  // namespace kccot

extern "C" {

int kccot_mixed_sqdist_partials(const float* real, const float* fake, int nprob, int B, long long K, void* ws,
                                size_t ws_bytes, int flags, void* stream) {
  if (int rc = check_common(nprob, B, B, K)) return rc;
  KCCOT_CHECK_ARG(real && fake && ws, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const bool tc_ok = (real != fake) && tc_sqdist_supported(real, fake, B, B, K);
  const int path = pick_path(flags, tc_ok);
  if (path < 0) {
    set_error("tcgen05 path requested but unsupported for B=%d K=%lld", B, K);
    return KCCOT_EUNSUPPORTED;
  }
  if (path == KCCOT_PATH_TCGEN05) {
    int ks, kbps;
    tc_sqdist_plan(nprob, 2 * B, K, &ks, &kbps);
    KCCOT_CHECK_ARG(ws_bytes >= (size_t)nprob * ks * kTcTile * 4, "workspace too small");
    return launch_sqdist_partials_tc(real, fake, nprob, B, B, K, ks, kbps, (float*)ws, st);
  }
  int ks;
  long long slab;
  choose_ksplit_simt(nprob, B, B, K, &ks, &slab);
  const size_t one = align_up((size_t)nprob * ks * B * B * 4, 256);
  KCCOT_CHECK_ARG(ws_bytes >= 3 * one, "workspace too small");
  const float* xs[3] = {real, real, fake};
  const float* ys[3] = {fake, real, fake};
  for (int q = 0; q < 3; ++q)
    if (int rc = launch_sqdist_partials_simt(xs[q], ys[q], nprob, B, B, K, ks, slab, (float*)((char*)ws + q * one), st))
      return rc;
  return KCCOT_OK;
}

size_t kccot_cost_bwd_workspace_bytes(int nprob, int Bx, int By, long long K) {
  if (nprob < 1 || Bx < 1 || By < 1 || K < 1) return 0;
  if (large_path_wanted(Bx, By, false)) return large_cost_bwd_ws_bytes(Bx, By, K, false);
  return align_up((Bx + By <= 128 ? tc_grad_ws_bytes(nprob) : 0) + 256, 256);
}

int kccot_cost_bwd(const float* Cbar, const float* x, const float* y, int nprob, int Bx, int By, long long K, float s,
                   float* gx, float* gy, void* ws, size_t ws_bytes, int flags, void* stream) {
  if (int rc = check_common(nprob, Bx, By, K)) return rc;
  KCCOT_CHECK_ARG(Cbar && x && y, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int acc = (flags & KCCOT_FLAG_ACCUMULATE) ? 1 : 0;
  const long long cprob = (long long)Bx * By;
  if ((flags & 3) != KCCOT_PATH_SIMT && large_path_wanted(Bx, By, false) && ws &&
      ws_bytes >= large_cost_bwd_ws_bytes(Bx, By, K, false)) {
    for (int p = 0; p < nprob; ++p)
      if (int rc = large_cost_bwd(Cbar + p * cprob, x + (long long)p * Bx * K, y + (long long)p * By * K, Bx, By, K, s,
                                  gx ? gx + (long long)p * Bx * K : nullptr, gy ? gy + (long long)p * By * K : nullptr, acc, ws,
                                  ws_bytes, st))
        return rc;
    return KCCOT_OK;
  }
  const bool tc_ok = (flags & 3) != KCCOT_PATH_SIMT && x != y && gx != gy && ws &&
                     ws_bytes >= tc_grad_ws_bytes(nprob) && tc_grad_supported(x, y, Bx, By, K, gx, gy);
  if ((flags & 3) == KCCOT_PATH_TCGEN05 && !tc_ok) {
    set_error("tcgen05 gradient path requested but unsupported for Bx=%d By=%d K=%lld", Bx, By, K);
    return KCCOT_EUNSUPPORTED;
  }
  if (tc_ok) return launch_grad_pair_tc(Cbar, x, y, nprob, Bx, By, K, s, gx, gy, acc, (float*)ws, st);
  if (gx)
    if (int rc = launch_cost_bwd_simt(Cbar, By, 1, cprob, x, y, nprob, Bx, By, K, s, gx, acc, st)) return rc;
  if (gy)
    if (int rc = launch_cost_bwd_simt(Cbar, 1, By, cprob, y, x, nprob, By, Bx, K, s, gy, acc || (gy == gx), st))
      return rc;
  return KCCOT_OK;
}

int kccot_martingale_bwd(const float* Cbar, const float* h, const float* M, int nprob, int Bx, int By, int T, int J,
                         float s, float* gh, float* gM, int flags, void* stream) {
  KCCOT_CHECK_ARG(Cbar && h && M, "null pointer");
  KCCOT_CHECK_ARG(nprob >= 1 && Bx >= 1 && By >= 1 && T >= 2 && J >= 1, "bad sizes");
  const int acc = (flags & KCCOT_FLAG_ACCUMULATE) ? 1 : 0;
  return launch_martingale_bwd(Cbar, (long long)Bx * By, h, M, nprob, Bx, By, T, J, s, 1.f, gh, gM, acc, acc,
                               (cudaStream_t)stream);
}

size_t kccot_mixed_cost_bwd_workspace_bytes(int nprob, int B, long long K) {
  if (nprob < 1 || B < 1 || K < 1) return 0;
  if (large_path_wanted(B, B, false)) return large_cost_bwd_ws_bytes(B, B, K, true);
  return align_up((2 * B <= 128 ? tc_grad_ws_bytes(nprob) : 0) + 256, 256);
}

int kccot_mixed_cost_bwd(const float* Cbar3, const float* real, const float* fake, int nprob, int B, long long K,
                         const float* h_fake, const float* m_real, const float* h_real, const float* m_fake, int T,
                         int J, float s, float* g_real, float* g_fake, float* gh_fake, float* gm_real, float* gh_real,
                         float* gm_fake, void* ws, size_t ws_bytes, int flags, void* stream) {
  if (int rc = check_common(nprob, B, B, K)) return rc;
  KCCOT_CHECK_ARG(Cbar3 && real && fake && h_fake && m_real && h_real && m_fake, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int acc = (flags & KCCOT_FLAG_ACCUMULATE) ? 1 : 0;
  const long long BB = (long long)B * B, cprob = 3 * BB;
  const float* Cxy = Cbar3;
  const float* Cxx = Cbar3 + BB;
  const float* Cyy = Cbar3 + 2 * BB;
  const bool want_tc = (flags & 3) != KCCOT_PATH_SIMT;
  const bool tc_ok = want_tc && (real != fake) && tc_grad_supported(real, fake, B, B, K, g_real, g_fake) && ws &&
                     ws_bytes >= tc_grad_ws_bytes(nprob);
  if ((flags & 3) == KCCOT_PATH_TCGEN05 && !tc_ok) {
    set_error("tcgen05 gradient path requested but unsupported for B=%d K=%lld", B, K);
    return KCCOT_EUNSUPPORTED;
  }
  // martingale terms: one launch
  const MartJobs jobs = mixed_mart_jobs(Cbar3, B, h_fake, m_real, h_real, m_fake, gh_fake, gm_real, gh_real, gm_fake, acc);
  if (want_tc && real != fake && large_path_wanted(B, B, false) && ws && ws_bytes >= large_cost_bwd_ws_bytes(B, B, K, true)) {
    if (int rc = launch_martingale_jobs(jobs, 4, nprob, T, J, s, st)) return rc;
    for (int p = 0; p < nprob; ++p)
      if (int rc = large_mixed_cost_bwd(Cbar3 + p * cprob, real + (long long)p * B * K, fake + (long long)p * B * K, B, K, s,
                                        g_real ? g_real + (long long)p * B * K : nullptr,
                                        g_fake ? g_fake + (long long)p * B * K : nullptr, acc, ws, ws_bytes, st))
        return rc;
    return KCCOT_OK;
  }
  if (tc_ok)
    return mart_beside_grad(jobs, nprob, T, J, s, st, [&] {
      return launch_grad_tc(Cbar3, real, fake, nprob, B, B, K, s, g_real, g_fake, acc, (float*)ws, st);
    });
  if (g_fake) {
    if (int rc = launch_cost_bwd_simt(Cxy, 1, B, cprob, fake, real, nprob, B, B, K, s, g_fake, acc, st)) return rc;
    if (int rc = launch_cost_bwd_simt(Cyy, B, 1, cprob, fake, fake, nprob, B, B, K, s, g_fake, 1, st)) return rc;
    if (int rc = launch_cost_bwd_simt(Cyy, 1, B, cprob, fake, fake, nprob, B, B, K, s, g_fake, 1, st)) return rc;
  }
  if (g_real) {
    if (int rc = launch_cost_bwd_simt(Cxy, B, 1, cprob, real, fake, nprob, B, B, K, s, g_real, acc, st)) return rc;
    if (int rc = launch_cost_bwd_simt(Cxx, B, 1, cprob, real, real, nprob, B, B, K, s, g_real, 1, st)) return rc;
    if (int rc = launch_cost_bwd_simt(Cxx, 1, B, cprob, real, real, nprob, B, B, K, s, g_real, 1, st)) return rc;
  }
  if (int rc = launch_martingale_jobs(jobs, 4, nprob, T, J, s, st)) return rc;
  return KCCOT_OK;
}

}  // extern "C"
