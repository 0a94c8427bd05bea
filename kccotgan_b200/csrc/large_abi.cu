// Orchestration of the large-batch cost path (stacked rows > 128, i.e. B > 64 for the mixed loss): workspace
// carving and the launch sequences around gemm_f16x3.cu.  Called from the C-ABI entry points in cost_abi.cu;
// no allocation, no synchronisation.  Reference arithmetic: gan_utils.py:14-17, :34-38 and their adjoints.
#include "cost.cuh"
#include "large.cuh"

namespace kccot {

namespace {
struct Carver {
  char* base;
  size_t off = 0;
  explicit Carver(void* p) : base((char*)p) {}
  template <typename T>
  T* take(size_t count) {
    off = align_up(off, 256);
    T* r = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += count * sizeof(T);
    return r;
  }
};

long long pad64(long long v) { return (v + 63) / 64 * 64; }

int stats_segments(int R, long long K) {
  const long long ccta = (K + 127) / 128;
  long long nseg = (2048 + ccta - 1) / ccta;
  const long long cap = (R + 31) / 32 < 32 ? (R + 31) / 32 : 32;
  if (nseg > cap) nseg = cap;
  return (int)(nseg < 1 ? 1 : nseg);
}

struct FwdWs {
  float *scal, *part, *mean, *norms;
  __half *Zh1, *Zh2;
  float* P[3];
  int ksplit, kb_per_split, nseg;
  long long Kp;
  G3Job job[3];
  int njobs;
  size_t bytes;
};

// blocks: mixed = (xy, xx, yy) over Z = [real; fake]; pair = (xy) over Z = [x; y]; same = (xx) over Z = x
FwdWs carve_fwd(void* ws, int Bx, int By, long long K, bool same, bool mixed) {
  FwdWs w{};
  const int R = same ? Bx : Bx + By;
  w.Kp = pad64(K);
  w.nseg = stats_segments(R, K);
  w.njobs = mixed ? 3 : 1;
  if (mixed) {
    w.job[0] = G3Job{0, Bx, Bx, By, 0, 0, 0, 0, nullptr, By, 0};
    w.job[1] = G3Job{0, 0, Bx, Bx, 0, 0, 0, 1, nullptr, Bx, 0};
    w.job[2] = G3Job{Bx, Bx, By, By, 0, 0, 0, 1, nullptr, By, 0};
  } else if (same) {
    w.job[0] = G3Job{0, 0, Bx, Bx, 0, 0, 0, 1, nullptr, Bx, 0};
  } else {
    w.job[0] = G3Job{0, Bx, Bx, By, 0, 0, 0, 0, nullptr, By, 0};
  }
  int ntiles = 0;
  for (int j = 0; j < w.njobs; ++j) ntiles += g3_count_tiles_pair(&w.job[j]);
  g3_plan_split(ntiles, (int)(w.Kp / G3_BK), num_sms() / 2, &w.ksplit, &w.kb_per_split);
  Carver c(ws);
  w.scal = c.take<float>(kScalCount);
  w.part = c.take<float>((size_t)w.nseg * K);
  w.mean = c.take<float>((size_t)w.Kp);
  w.norms = c.take<float>((size_t)R);
  w.Zh1 = c.take<__half>((size_t)R * w.Kp);
  w.Zh2 = c.take<__half>((size_t)R * w.Kp);
  for (int j = 0; j < w.njobs; ++j) {
    w.job[j].ks_stride = (long long)w.job[j].m * w.job[j].ld;
    w.P[j] = c.take<float>((size_t)w.ksplit * w.job[j].ks_stride);
    w.job[j].out = w.P[j];
  }
  w.bytes = align_up(c.off, 256);
  return w;
}

struct BwdWs {
  float *scal, *part, *mean, *Wtmp, *rs_part, *rowsum;
  __half *ZT1, *ZT2, *Wh1, *Wh2;
  int nseg, Rp;
  long long Kp;
  size_t bytes;
};

BwdWs carve_bwd(void* ws, int Bx, int By, long long K) {
  BwdWs w{};
  const int R = Bx + By;
  const int maxrows = Bx > By ? Bx : By;
  w.Kp = pad64(K);
  w.Rp = (int)pad64(R);
  w.nseg = stats_segments(R, K);
  Carver c(ws);
  w.scal = c.take<float>(kScalCount);
  w.part = c.take<float>((size_t)w.nseg * K);
  w.mean = c.take<float>((size_t)w.Kp);
  w.ZT1 = c.take<__half>((size_t)w.Kp * w.Rp);
  w.ZT2 = c.take<__half>((size_t)w.Kp * w.Rp);
  w.Wtmp = c.take<float>((size_t)maxrows * w.Rp);
  w.rs_part = c.take<float>((size_t)((R + 31) / 32) * maxrows);
  w.rowsum = c.take<float>((size_t)maxrows);
  w.Wh1 = c.take<__half>((size_t)maxrows * w.Rp);
  w.Wh2 = c.take<__half>((size_t)maxrows * w.Rp);
  w.bytes = align_up(c.off, 256);
  return w;
}

int run_fwd(const FwdWs& w, const float* x, const float* y, int Bx, int By, long long K, bool same, cudaStream_t st) {
  const int R = same ? Bx : Bx + By;
  if (int rc = large_launch_stats(x, same ? nullptr : y, Bx, same ? 0 : By, K, w.nseg, w.part, w.mean, w.scal, st)) return rc;
  if (int rc = large_launch_split(x, same ? nullptr : y, Bx, same ? 0 : By, K, w.Kp, 0, w.mean, w.scal, w.Zh1, w.Zh2, nullptr,
                                  nullptr, st))
    return rc;
  if (int rc = large_launch_rownorm(w.Zh1, w.Zh2, R, K, w.Kp, w.norms, st)) return rc;
  G3Params P{};
  for (int j = 0; j < w.njobs; ++j) P.job[j] = w.job[j];
  P.njobs = w.njobs;
  P.ksplit = w.ksplit;
  P.kb_per_split = w.kb_per_split;
  P.alpha = 1.f;
  P.alpha_dev = nullptr;
  return launch_gemm_f16x3_pair(w.Zh1, w.Zh2, R, w.Kp, w.Zh1, w.Zh2, R, w.Kp, K, P, st);
}

int run_bwd_rows(const BwdWs& w, const float* Cxx, const float* Cxy, const float* Cyy, int Bx, int By, long long K, float s,
                 int row_off, int nrows, float* g, int accumulate, cudaStream_t st) {
  const int R = Bx + By;
  if (int rc = large_launch_wbuild(Cxx, Cxy, Cyy, Bx, By, row_off, nrows, w.Rp, w.Wtmp, w.rs_part, w.rowsum, w.scal, w.Wh1,
                                   w.Wh2, st))
    return rc;
  G3Params P{};
  P.job[0] = G3Job{0, 0, nrows, (int)K, 0, 0, 0, 0, g, K, 0};
  g3_count_tiles_pair(&P.job[0]);
  P.njobs = 1;
  P.ksplit = 1;
  P.kb_per_split = (int)(w.Rp / G3_BK);
  P.alpha = -2.f * s;
  P.alpha_dev = w.scal + kScalGradAlpha;
  P.accumulate = accumulate;
  return launch_gemm_f16x3_pair(w.Wh1, w.Wh2, nrows, w.Rp, w.ZT1, w.ZT2, K, w.Rp, R, P, st);
}
}  // namespace

bool large_path_wanted(int Bx, int By, bool same) { return (same ? Bx : Bx + By) > 128; }

size_t large_cost_fwd_ws_bytes(int Bx, int By, long long K, bool same, bool mixed) {
  return carve_fwd(nullptr, Bx, By, K, same, mixed).bytes;
}
size_t large_cost_bwd_ws_bytes(int Bx, int By, long long K, bool mixed) {
  (void)mixed;
  return carve_bwd(nullptr, Bx, By, K).bytes;
}

int large_mixed_cost_fwd(const float* real, const float* fake, int B, long long K, const float* h_fake,
                         const float* m_real, const float* h_real, const float* m_fake, int T, int J, float s,
                         float* C3, void* ws, size_t ws_bytes, cudaStream_t st) {
  KCCOT_CHECK_ARG(K < (1LL << 31) - 64 && (long long)B * 2 < (1LL << 30), "sizes beyond the large path's 32-bit tile coordinates");
  const FwdWs w = carve_fwd(ws, B, B, K, false, true);
  KCCOT_CHECK_ARG(ws_bytes >= w.bytes, "workspace too small (large-batch cost path needs %zu bytes, got %zu)", w.bytes, ws_bytes);
  if (int rc = run_fwd(w, real, fake, B, B, K, false, st)) return rc;
  const long long BB = (long long)B * B;
  LargeFin F{};
  // order xy, xx, yy — gan_utils.py:221-223
  F.b[0] = LargeFinBlock{w.P[0], B, w.job[0].ks_stride, w.ksplit, 0, w.norms, w.norms + B, h_fake, m_real, nullptr, nullptr,
                         C3, B, B, B, 0, 0};
  F.b[1] = LargeFinBlock{w.P[1], B, w.job[1].ks_stride, w.ksplit, 1, w.norms, w.norms, h_real, m_real, nullptr, nullptr,
                         C3 + BB, B, B, B, 1, 0};
  F.b[2] = LargeFinBlock{w.P[2], B, w.job[2].ks_stride, w.ksplit, 1, w.norms + B, w.norms + B, h_fake, m_fake, nullptr,
                         nullptr, C3 + 2 * BB, B, B, B, 1, 0};
  return large_launch_finalize(F, 3, T, J, s, w.scal, st);
}

int large_cost_fwd(const float* x, const float* y, int Bx, int By, long long K, const float* h1, const float* M1,
                   const float* h2, const float* M2, int T, int J, float s, float* C, void* ws, size_t ws_bytes,
                   cudaStream_t st) {
  KCCOT_CHECK_ARG(K < (1LL << 31) - 64 && (long long)Bx + By < (1LL << 30), "sizes beyond the large path's 32-bit tile coordinates");
  const bool same = (x == y);
  const FwdWs w = carve_fwd(ws, Bx, By, K, same, false);
  KCCOT_CHECK_ARG(ws_bytes >= w.bytes, "workspace too small (large-batch cost path needs %zu bytes, got %zu)", w.bytes, ws_bytes);
  if (int rc = run_fwd(w, x, y, Bx, By, K, same, st)) return rc;
  LargeFin F{};
  F.b[0] = LargeFinBlock{w.P[0], By, w.job[0].ks_stride, w.ksplit, same ? 1 : 0, w.norms, same ? w.norms : w.norms + Bx,
                         h1, M1, h2, M2, C, By, Bx, By, same ? 1 : 0, 0};
  return large_launch_finalize(F, 1, T, J, s, w.scal, st);
}

int large_mixed_cost_bwd(const float* Cbar3, const float* real, const float* fake, int B, long long K, float s,
                         float* g_real, float* g_fake, int accumulate, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (!g_real && !g_fake) return KCCOT_OK;
  const BwdWs w = carve_bwd(ws, B, B, K);
  KCCOT_CHECK_ARG(ws_bytes >= w.bytes, "workspace too small (large-batch adjoint needs %zu bytes, got %zu)", w.bytes, ws_bytes);
  if (int rc = large_launch_stats(real, fake, B, B, K, w.nseg, w.part, w.mean, w.scal, st)) return rc;
  if (int rc = large_launch_split(real, fake, B, B, K, w.Kp, w.Rp, w.mean, w.scal, nullptr, nullptr, w.ZT1, w.ZT2, st)) return rc;
  const long long BB = (long long)B * B;
  const float *Cxy = Cbar3, *Cxx = Cbar3 + BB, *Cyy = Cbar3 + 2 * BB;
  if (g_fake)
    if (int rc = run_bwd_rows(w, Cxx, Cxy, Cyy, B, B, K, s, B, B, g_fake, accumulate, st)) return rc;
  if (g_real)
    if (int rc = run_bwd_rows(w, Cxx, Cxy, Cyy, B, B, K, s, 0, B, g_real, accumulate, st)) return rc;
  return KCCOT_OK;
}

int large_cost_bwd(const float* Cbar, const float* x, const float* y, int Bx, int By, long long K, float s, float* gx,
                   float* gy, int accumulate, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (!gx && !gy) return KCCOT_OK;
  const BwdWs w = carve_bwd(ws, Bx, By, K);
  KCCOT_CHECK_ARG(ws_bytes >= w.bytes, "workspace too small (large-batch adjoint needs %zu bytes, got %zu)", w.bytes, ws_bytes);
  if (int rc = large_launch_stats(x, y, Bx, By, K, w.nseg, w.part, w.mean, w.scal, st)) return rc;
  if (int rc = large_launch_split(x, y, Bx, By, K, w.Kp, w.Rp, w.mean, w.scal, nullptr, nullptr, w.ZT1, w.ZT2, st)) return rc;
  if (gx)
    if (int rc = run_bwd_rows(w, nullptr, Cbar, nullptr, Bx, By, K, s, 0, Bx, gx, accumulate, st)) return rc;
  if (gy)   // gx == gy (x and y are the same tensor): the second product adds to the first
    if (int rc = run_bwd_rows(w, nullptr, Cbar, nullptr, Bx, By, K, s, Bx, By, gy, accumulate || gy == gx, st)) return rc;
  return KCCOT_OK;
}

// ------------------------------------------------------------------------------------------------
// Row shards of ONE large problem (BASELINE config 5 on N GPUs).  Inputs (videos, h, M) are replicated; this rank
// owns the samples [row0, row0 + Brows) and computes the cost ROWS of the three blocks, later the gradient rows.
// The workspace of the forward call carries the transposed split and the scales to the backward call.
// ------------------------------------------------------------------------------------------------
namespace {
// Column layout of the shared-context split (large.cuh): nc context columns padded to Kcp, then nq predicted columns
// padded to Kqp
struct CtxCols {
  int period, clen, nc, nq, Kcp, Kqp;
  CtxCols(long long K, long long p, long long l)
      : period((int)p), clen((int)l), nc((int)(K / p * l)), nq((int)(K - K / p * l)), Kcp((int)pad64(nc)),
        Kqp((int)pad64(nq)) {}
};

struct ShardWs {
  float *scal, *part, *mean, *norms, *Wtmp, *rs_part, *rowsum;
  __half *Zh1, *Zh2, *ZT1, *ZT2, *Wh1, *Wh2;
  float* P[3];
  float* g_pred;           // shared-context hint only: the adjoint GEMM's [Brows][nq] predicted-column rows
  int nseg, Rp;
  long long Kp;            // pitch of the split (padded permuted width under the hint)
  size_t bytes;
};
ShardWs carve_shard(void* ws, int B, long long K, int Brows, const CtxCols* cc = nullptr) {
  ShardWs w{};
  const int R = 2 * B;
  w.Kp = cc ? (long long)cc->Kcp + cc->Kqp : pad64(K);
  w.Rp = (int)pad64(R);
  w.nseg = stats_segments(R, K);
  Carver c(ws);
  w.scal = c.take<float>(kScalCount);
  w.part = c.take<float>((size_t)w.nseg * K);
  w.mean = c.take<float>((size_t)w.Kp);
  w.norms = c.take<float>((size_t)R);
  w.Zh1 = c.take<__half>((size_t)R * w.Kp);
  w.Zh2 = c.take<__half>((size_t)R * w.Kp);
  w.ZT1 = c.take<__half>((size_t)w.Kp * w.Rp);
  w.ZT2 = c.take<__half>((size_t)w.Kp * w.Rp);
  for (int q = 0; q < 3; ++q) w.P[q] = c.take<float>((size_t)Brows * B);
  w.Wtmp = c.take<float>((size_t)Brows * w.Rp);
  w.rs_part = c.take<float>((size_t)((R + 31) / 32) * Brows);
  w.rowsum = c.take<float>((size_t)Brows);
  w.Wh1 = c.take<__half>((size_t)Brows * w.Rp);
  w.Wh2 = c.take<__half>((size_t)Brows * w.Rp);
  if (cc) w.g_pred = c.take<float>((size_t)Brows * cc->nq);
  w.bytes = align_up(c.off, 256);
  return w;
}
}  // namespace

size_t large_shard_ws_bytes(int B, long long K, int Brows) { return carve_shard(nullptr, B, K, Brows).bytes; }
size_t large_shard_ws_bytes_ctx(int B, long long K, int Brows, long long period, long long clen) {
  const CtxCols cc(K, period, clen);
  return carve_shard(nullptr, B, K, Brows, &cc).bytes;
}

namespace {
// Video element type V (float, or bf16 bits): only the pre-pass reads the videos, so only it depends on V.
// cc != nullptr: the shared-context hint (large.cuh) — the context columns' Gram is computed once, real rows x all
// reals, and the three blocks add their predicted columns' Gram to it.
template <typename V>
int shard_cost_fwd(const V* real, const V* fake, int B, long long K, int row0, int Brows, const float* h_fake,
                   const float* m_real, const float* h_real, const float* m_fake, int T, int J, float s, float* C3rows,
                   void* ws, size_t ws_bytes, cudaStream_t st, const CtxCols* cc = nullptr) {
  KCCOT_CHECK_ARG(row0 >= 0 && Brows >= 1 && row0 + Brows <= B, "bad row range [%d, %d) of %d", row0, row0 + Brows, B);
  const ShardWs w = carve_shard(ws, B, K, Brows, cc);
  KCCOT_CHECK_ARG(ws_bytes >= w.bytes, "workspace too small (row-shard cost path needs %zu bytes, got %zu)", w.bytes, ws_bytes);
  const int R = 2 * B;
  if (cc) {
    if (int rc = large_launch_stats_ctx(real, fake, B, K, cc->period, cc->clen, w.nseg, w.part, w.mean, w.scal, st)) return rc;
    if (int rc = large_launch_split_ctx(real, fake, B, K, cc->period, cc->clen, cc->Kcp, w.Kp, w.Rp, w.mean, w.scal, w.Zh1,
                                        w.Zh2, w.ZT1, w.ZT2, st))
      return rc;
    if (int rc = large_launch_rownorm(w.Zh1, w.Zh2, R, w.Kp, w.Kp, w.norms, st)) return rc;
  } else {
    if (int rc = large_launch_stats(real, fake, B, B, K, w.nseg, w.part, w.mean, w.scal, st)) return rc;
    if (int rc = large_launch_split(real, fake, B, B, K, w.Kp, w.Rp, w.mean, w.scal, w.Zh1, w.Zh2, w.ZT1, w.ZT2, st)) return rc;
    if (int rc = large_launch_rownorm(w.Zh1, w.Zh2, R, K, w.Kp, w.norms, st)) return rc;
  }
  G3Params P{};
  // xy: real rows x all fakes; xx: real rows x all reals; yy: fake rows x all fakes (no symmetry across ranks)
  P.job[0] = G3Job{row0, B, Brows, B, 0, 0, 0, 0, w.P[0], B, 0};
  P.job[1] = G3Job{row0, 0, Brows, B, 0, 0, 0, 0, w.P[1], B, 0};
  P.job[2] = G3Job{B + row0, B, Brows, B, 0, 0, 0, 0, w.P[2], B, 0};
  P.njobs = 3;
  for (int j = 0; j < 3; ++j) g3_count_tiles_pair(&P.job[j]);
  P.ksplit = 1;
  P.kb_per_split = (int)(w.Kp / G3_BK);
  P.alpha = 1.f;
  if (cc) {
    // context columns: real and fake rows are the same there, so the three blocks share real rows x all reals
    G3Params Pc{};
    Pc.job[0] = P.job[1];
    g3_count_tiles_pair(&Pc.job[0]);
    Pc.njobs = 1;
    Pc.ksplit = 1;
    Pc.kb_per_split = cc->Kcp / G3_BK;
    Pc.alpha = 1.f;
    if (int rc = launch_gemm_f16x3_pair(w.Zh1, w.Zh2, R, w.Kp, w.Zh1, w.Zh2, R, w.Kp, cc->nc, Pc, st)) return rc;
    const size_t pb = (size_t)Brows * B * sizeof(float);
    KCCOT_CUDA(cudaMemcpyAsync(w.P[0], w.P[1], pb, cudaMemcpyDeviceToDevice, st));
    KCCOT_CUDA(cudaMemcpyAsync(w.P[2], w.P[1], pb, cudaMemcpyDeviceToDevice, st));
    // predicted columns: the three blocks, added to it
    P.kb_per_split = cc->Kqp / G3_BK;
    P.accumulate = 1;
    if (int rc = launch_gemm_f16x3_pair(w.Zh1 + cc->Kcp, w.Zh2 + cc->Kcp, R, w.Kp, w.Zh1 + cc->Kcp, w.Zh2 + cc->Kcp, R, w.Kp,
                                        cc->nq, P, st))
      return rc;
  } else {
    if (int rc = launch_gemm_f16x3_pair(w.Zh1, w.Zh2, R, w.Kp, w.Zh1, w.Zh2, R, w.Kp, K, P, st)) return rc;
  }
  const long long RB = (long long)Brows * B, hm = (long long)T * J;
  LargeFin F{};
  F.b[0] = LargeFinBlock{w.P[0], B, RB, 1, 0, w.norms + row0, w.norms + B, h_fake + row0 * hm, m_real, nullptr, nullptr,
                         C3rows, B, Brows, B, 0, 0};
  F.b[1] = LargeFinBlock{w.P[1], B, RB, 1, 0, w.norms + row0, w.norms, h_real + row0 * hm, m_real, nullptr, nullptr,
                         C3rows + RB, B, Brows, B, 1, row0};
  F.b[2] = LargeFinBlock{w.P[2], B, RB, 1, 0, w.norms + B + row0, w.norms + B, h_fake + row0 * hm, m_fake, nullptr, nullptr,
                         C3rows + 2 * RB, B, Brows, B, 1, row0};
  return large_launch_finalize(F, 3, T, J, s, w.scal, st);
}

// Gradient element type G (float, or bf16 bits): only the adjoint GEMM's store depends on G.
template <typename G>
int shard_cost_bwd(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B, long long K, int row0, int Brows,
                   const float* h_fake, const float* m_real, const float* h_real, const float* m_fake, int T, int J,
                   float s, G* g_fake_rows, float* gh_fake_rows, float* gm_real_part, float* gh_real_rows,
                   float* gm_fake_part, void* ws, size_t ws_bytes, cudaStream_t st, const CtxCols* cc = nullptr) {
  const ShardWs w = carve_shard(ws, B, K, Brows, cc);
  KCCOT_CHECK_ARG(ws_bytes >= w.bytes, "workspace too small (row-shard cost path needs %zu bytes, got %zu)", w.bytes, ws_bytes);
  const long long RB = (long long)Brows * B, hm = (long long)T * J;
  const float *Cxy = Cbar3rows, *Cxx = Cbar3rows + RB, *Cyy = Cbar3rows + 2 * RB;
  // martingale adjoints (gan_utils.py:34-38): h gradients belong to the row samples (local), M gradients to the
  // column samples (partial over this rank's rows)
  MartJobs jobs{};
  jobs.j[0] = MartJob{gh_fake_rows, Cxy, m_real, Cyy, m_fake, 0, B, Brows, B, 0, 0, 0};
  jobs.j[1] = MartJob{gm_real_part, Cxy, h_fake + row0 * hm, Cxx, h_real + row0 * hm, 0, B, B, Brows, 1, 1, 0};
  jobs.j[2] = MartJob{gh_real_rows, Cxx, m_real, nullptr, nullptr, 0, B, Brows, B, 0, 0, 0};
  jobs.j[3] = MartJob{gm_fake_part, Cyy, h_fake + row0 * hm, nullptr, nullptr, 0, B, B, Brows, 1, 1, 0};
  if (int rc = launch_martingale_jobs(jobs, 4, 1, T, J, s, st)) return rc;
  if (!g_fake_rows) return KCCOT_OK;
  if (int rc = large_launch_wbuild_shard(XYcol, YYcol, Cyy, B, B, row0, Brows, w.Rp, w.Wtmp, w.rs_part, w.rowsum, w.scal,
                                         w.Wh1, w.Wh2, st))
    return rc;
  G3Params P{};
  P.job[0] = G3Job{0, 0, Brows, (int)K, 0, 0, 0, 0, reinterpret_cast<float*>(g_fake_rows), K, 0};
  if (cc) {
    // the predicted columns only (rows [Kcp, Kcp + nq) of ZT) into g_pred, then back to the video columns
    P.job[0] = G3Job{0, 0, Brows, cc->nq, 0, 0, 0, 0, w.g_pred, cc->nq, 0};
    g3_count_tiles_pair(&P.job[0]);
    P.njobs = 1;
    P.ksplit = 1;
    P.kb_per_split = (int)(w.Rp / G3_BK);
    P.alpha = -2.f * s;
    P.alpha_dev = w.scal + kScalGradAlpha;
    const long long zoff = (long long)cc->Kcp * w.Rp;
    const int R = 2 * B;
    int rc;
    if constexpr (sizeof(G) == 2)
      rc = launch_gemm_f16x3_pair_bf16(w.Wh1, w.Wh2, Brows, w.Rp, w.ZT1 + zoff, w.ZT2 + zoff, cc->nq, w.Rp, R, P, st);
    else
      rc = launch_gemm_f16x3_pair(w.Wh1, w.Wh2, Brows, w.Rp, w.ZT1 + zoff, w.ZT2 + zoff, cc->nq, w.Rp, R, P, st);
    if (rc) return rc;
    return large_launch_ctx_scatter(reinterpret_cast<const G*>(w.g_pred), Brows, (int)K, cc->period, cc->clen, g_fake_rows,
                                    st);
  }
  g3_count_tiles_pair(&P.job[0]);
  P.njobs = 1;
  P.ksplit = 1;
  P.kb_per_split = (int)(w.Rp / G3_BK);
  P.alpha = -2.f * s;
  P.alpha_dev = w.scal + kScalGradAlpha;
  const int R = 2 * B;
  if constexpr (sizeof(G) == 2)
    return launch_gemm_f16x3_pair_bf16(w.Wh1, w.Wh2, Brows, w.Rp, w.ZT1, w.ZT2, K, w.Rp, R, P, st);
  else
    return launch_gemm_f16x3_pair(w.Wh1, w.Wh2, Brows, w.Rp, w.ZT1, w.ZT2, K, w.Rp, R, P, st);
}
}  // namespace

int large_shard_cost_fwd(const float* real, const float* fake, int B, long long K, int row0, int Brows, const float* h_fake,
                         const float* m_real, const float* h_real, const float* m_fake, int T, int J, float s,
                         float* C3rows, void* ws, size_t ws_bytes, cudaStream_t st) {
  return shard_cost_fwd(real, fake, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s, C3rows, ws, ws_bytes, st);
}
int large_shard_cost_fwd(const uint16_t* real, const uint16_t* fake, int B, long long K, int row0, int Brows,
                         const float* h_fake, const float* m_real, const float* h_real, const float* m_fake, int T, int J,
                         float s, float* C3rows, void* ws, size_t ws_bytes, cudaStream_t st) {
  return shard_cost_fwd(real, fake, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s, C3rows, ws, ws_bytes, st);
}

// g_fake_rows [Brows][K]; gh_* rows [Brows][T][J] (own samples); gm_* partial sums [B][T][J] over this rank's rows
// (the caller all-reduces them).  `ws` is the workspace of the matching large_shard_cost_fwd call.
int large_shard_cost_bwd(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B, long long K, int row0,
                         int Brows, const float* h_fake, const float* m_real, const float* h_real, const float* m_fake,
                         int T, int J, float s, float* g_fake_rows, float* gh_fake_rows, float* gm_real_part,
                         float* gh_real_rows, float* gm_fake_part, void* ws, size_t ws_bytes, cudaStream_t st) {
  return shard_cost_bwd(Cbar3rows, XYcol, YYcol, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s, g_fake_rows,
                        gh_fake_rows, gm_real_part, gh_real_rows, gm_fake_part, ws, ws_bytes, st);
}
int large_shard_cost_bwd(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B, long long K, int row0,
                         int Brows, const float* h_fake, const float* m_real, const float* h_real, const float* m_fake,
                         int T, int J, float s, uint16_t* g_fake_rows, float* gh_fake_rows, float* gm_real_part,
                         float* gh_real_rows, float* gm_fake_part, void* ws, size_t ws_bytes, cudaStream_t st) {
  return shard_cost_bwd(Cbar3rows, XYcol, YYcol, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s, g_fake_rows,
                        gh_fake_rows, gm_real_part, gh_real_rows, gm_fake_part, ws, ws_bytes, st);
}

int large_shard_cost_fwd_ctx(const float* real, const float* fake, int B, long long K, int row0, int Brows,
                             const float* h_fake, const float* m_real, const float* h_real, const float* m_fake, int T,
                             int J, float s, float* C3rows, void* ws, size_t ws_bytes, long long period, long long clen,
                             cudaStream_t st) {
  const CtxCols cc(K, period, clen);
  return shard_cost_fwd(real, fake, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s, C3rows, ws, ws_bytes, st,
                        &cc);
}
int large_shard_cost_fwd_ctx(const uint16_t* real, const uint16_t* fake, int B, long long K, int row0, int Brows,
                             const float* h_fake, const float* m_real, const float* h_real, const float* m_fake, int T,
                             int J, float s, float* C3rows, void* ws, size_t ws_bytes, long long period, long long clen,
                             cudaStream_t st) {
  const CtxCols cc(K, period, clen);
  return shard_cost_fwd(real, fake, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s, C3rows, ws, ws_bytes, st,
                        &cc);
}
int large_shard_cost_bwd_ctx(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B, long long K, int row0,
                             int Brows, const float* h_fake, const float* m_real, const float* h_real,
                             const float* m_fake, int T, int J, float s, float* g_fake_rows, float* gh_fake_rows,
                             float* gm_real_part, float* gh_real_rows, float* gm_fake_part, void* ws, size_t ws_bytes,
                             long long period, long long clen, cudaStream_t st) {
  const CtxCols cc(K, period, clen);
  return shard_cost_bwd(Cbar3rows, XYcol, YYcol, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s, g_fake_rows,
                        gh_fake_rows, gm_real_part, gh_real_rows, gm_fake_part, ws, ws_bytes, st, &cc);
}
int large_shard_cost_bwd_ctx(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B, long long K, int row0,
                             int Brows, const float* h_fake, const float* m_real, const float* h_real,
                             const float* m_fake, int T, int J, float s, uint16_t* g_fake_rows, float* gh_fake_rows,
                             float* gm_real_part, float* gh_real_rows, float* gm_fake_part, void* ws, size_t ws_bytes,
                             long long period, long long clen, cudaStream_t st) {
  const CtxCols cc(K, period, clen);
  return shard_cost_bwd(Cbar3rows, XYcol, YYcol, B, K, row0, Brows, h_fake, m_real, h_real, m_fake, T, J, s, g_fake_rows,
                        gh_fake_rows, gm_real_part, gh_real_rows, gm_fake_part, ws, ws_bytes, st, &cc);
}

}  // namespace kccot
