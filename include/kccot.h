/*
 * kccot.h — C ABI of libkccot.so: the B200 (sm_100a) causal-OT loss path of KCCOT-GAN.
 *
 * The reference (neuripss2020/kccotgan) has no FFI: its loss path is a set of plain Python
 * functions over TensorFlow eager tensors (gan_utils.py, data_utils.py:478-586).  This header is
 * the boundary a maintainer binds instead: every entry point below replaces the arithmetic of the
 * reference function cited next to it.  The Python mirror of the reference interface
 * (kccotgan_b200/gan_utils.py, data_utils.py) calls these through ctypes; INTEGRATION.md shows
 * the stub for the reference's own TensorFlow training loop.
 *
 * Conventions
 *   - All pointers are DEVICE pointers to contiguous fp32 unless stated (the *_bf16 mixed-loss and
 *     smoothing entries take bf16 videos); the caller owns every
 *     buffer (inputs, outputs, saved state, workspace).  The library allocates nothing per call
 *     and keeps no pointer after return.
 *   - `stream` is a cudaStream_t passed as void*.  Calls only enqueue work; none synchronises.
 *   - Return 0 on success, a negative KCCOT_E* code otherwise; kccot_last_error() gives the text
 *     (thread-local).  There is no CPU fallback: without a CUDA device every compute call fails.
 *   - Videos are [B, ...] tensors flattened to rows of length K (any order of the trailing axes:
 *     the cost sums over all of them, gan_utils.py:14-17,216-220).  h / M are [B, T, J].
 *   - "nprob" batches independent problems along a leading axis of every tensor.
 */
#ifndef KCCOT_H_
#define KCCOT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KCCOT_VERSION 203
#define KCCOT_SHARD_FLAGS_PER_RANK 256

/* error codes */
#define KCCOT_OK 0
#define KCCOT_EINVAL (-1)   /* bad shape / null pointer / misaligned buffer  -> Python ValueError */
#define KCCOT_ECUDA (-2)    /* CUDA runtime / driver error                   -> Python RuntimeError */
#define KCCOT_EWORKSPACE (-3)
#define KCCOT_EUNSUPPORTED (-4)

/* kernel-path selection flags (shape-based AUTO is what the product uses; the explicit values
 * exist so that tests can check the tensor-core path against the CUDA-core path) */
#define KCCOT_PATH_AUTO 0
#define KCCOT_PATH_SIMT 1      /* fp32 CUDA-core kernels, direct (x-y)^2 form, any shape */
#define KCCOT_PATH_TCGEN05 2   /* TMA + tcgen05 3xTF32 kernels (needs K % 4 == 0, 16-B aligned rows) */
#define KCCOT_FLAG_ACCUMULATE 16  /* gradient outputs: add into the buffer instead of overwriting */

int kccot_version(void);
const char* kccot_last_error(void);
/* 0 if the current device is sm_100 (B200); KCCOT_EUNSUPPORTED otherwise. */
int kccot_device_check(void);
/* number of kernels this library has launched so far in this process (bench.py's gpu_launches) */
unsigned long long kccot_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Cost matrices — gan_utils.py:6-18 (cost_xy), :21-43 (modified_cost), :46-72 (bi_causal_...)
 *   C[p,i,j] = s * sum_k (x[p,i,k] - y[p,j,k])^2
 *            + s * sum_{t<T-1,c} h1[p,i,t,c] * (M1[p,j,t+1,c] - M1[p,j,t,c])      (if h1 != NULL)
 *            + s * sum_{t<T-1,c} h2[p,i,t,c] * (M2[p,j,t+1,c] - M2[p,j,t,c])      (if h2 != NULL)
 * x [nprob,Bx,K], y [nprob,By,K], h* [nprob,Bx,T,J], M* [nprob,By,T,J], C [nprob,Bx,By].
 * x == y (same pointer) marks a self-cost: the diagonal is exactly 0 as in the reference.
 * ------------------------------------------------------------------------------------------ */
size_t kccot_cost_workspace_bytes(int nprob, int Bx, int By, long long K);
int kccot_cost_fwd(const float* x, const float* y, int nprob, int Bx, int By, long long K,
                   const float* h1, const float* M1, const float* h2, const float* M2, int T, int J,
                   float s, float* C, void* ws, size_t ws_bytes, int flags, void* stream);

/* The three cost matrices of the mixed loss in one pass over the videos —
 * gan_utils.py:221-223: xy = (real,fake,h_fake,m_real), xx = (real,real,h_real,m_real),
 * yy = (fake,fake,h_fake,m_fake).  C3 [nprob,3,B,B] in the order xy, xx, yy. */
size_t kccot_mixed_cost_workspace_bytes(int nprob, int B, long long K);
int kccot_mixed_cost_fwd(const float* real, const float* fake, int nprob, int B, long long K,
                         const float* h_fake, const float* m_real, const float* h_real,
                         const float* m_fake, int T, int J, float s, float* C3, void* ws,
                         size_t ws_bytes, int flags, void* stream);

/* First half of kccot_mixed_cost_fwd on its own: only the split-K partial squared distances of the
 * stacked rows [real; fake] are written to the workspace (the HBM-bound pass over the videos).
 * Exposed so that the streaming kernel can be timed and profiled in isolation. */
int kccot_mixed_sqdist_partials(const float* real, const float* fake, int nprob, int B, long long K,
                                void* ws, size_t ws_bytes, int flags, void* stream);

/* Adjoint of the squared-distance part: gx[p,i,:] = 2s * sum_j Cbar[p,i,j] (x_i - y_j),
 * gy[p,j,:] = 2s * sum_i Cbar[p,i,j] (y_j - x_i).  gx / gy may be NULL (not needed). */
size_t kccot_cost_bwd_workspace_bytes(int nprob, int Bx, int By, long long K);
int kccot_cost_bwd(const float* Cbar, const float* x, const float* y, int nprob, int Bx, int By,
                   long long K, float s, float* gx, float* gy, void* ws, size_t ws_bytes, int flags,
                   void* stream);
/* Adjoint of one martingale term: gh[:, :-1] = s*Cbar@DeltaM, gh[:, -1] = 0; gM from s*Cbar^T@h. */
int kccot_martingale_bwd(const float* Cbar, const float* h, const float* M, int nprob, int Bx, int By,
                         int T, int J, float s, float* gh, float* gM, int flags, void* stream);
/* Adjoint of kccot_mixed_cost_fwd.  Cbar3 [nprob,3,B,B] already carries the 2,-1,-1 weights and
 * the upstream gradient.  g_real may be NULL (data needs no gradient, kernel_train.py:289). */
size_t kccot_mixed_cost_bwd_workspace_bytes(int nprob, int B, long long K);
int kccot_mixed_cost_bwd(const float* Cbar3, const float* real, const float* fake, int nprob, int B,
                         long long K, const float* h_fake, const float* m_real, const float* h_real,
                         const float* m_fake, int T, int J, float s, float* g_real, float* g_fake,
                         float* gh_fake, float* gm_real, float* gh_real, float* gm_fake, void* ws,
                         size_t ws_bytes, int flags, void* stream);

/* ------------------------------------------------------------------------------------------
 * Log-domain Sinkhorn — gan_utils.py:138-165 (compute_sinkhorn), :86-121 (benchmark_sinkhorn)
 * nsolve independent B x B problems.  L iterations of the u / v updates with uniform marginals;
 * after iteration n (1-based) the solve stops if thresh > sum|u - u_prev| and
 * (exit_on_index ? n-1 >= Lmin : n >= Lmin)   [:159 vs :116].  The test runs on the device.
 * Saved for the backward (internal units: potentials * log2(e)/eps, cost shifted by its minimum):
 *   u_hist, v_hist [nsolve, L+1, B];  nits [nsolve] int32;  cost [nsolve] = sum(pi * C).
 * ------------------------------------------------------------------------------------------ */
size_t kccot_sinkhorn_workspace_bytes(int nsolve, int B, int L);
int kccot_sinkhorn_fwd(const float* C, int nsolve, int B, float eps, int L, int Lmin, float thresh,
                       int exit_on_index, float* u_hist, float* v_hist, int32_t* nits, float* cost,
                       void* ws, size_t ws_bytes, void* stream);
/* Reverse mode through the executed iterations (the reference has no stop_gradient; TF's tape
 * unrolls the loop).  Cbar[n] = gcost[n] * d cost[n] / d C[n].  gcost [nsolve] on the device. */
int kccot_sinkhorn_bwd(const float* C, int nsolve, int B, float eps, int L, const float* u_hist,
                       const float* v_hist, const int32_t* nits, const float* gcost, float* Cbar,
                       void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Row-sharded mixed loss, fused exchange (BASELINE config 5 on N GPUs).  Videos, h and M are replicated on
 * every rank (or all-gathered once by the caller); this rank owns the samples [row0, row0 + Brows): it
 * computes the cost ROWS of the xy, xx, yy blocks (C3rows [3,Brows,B]), runs its row block of the three
 * Sinkhorn solves inside ONE persistent kernel that exchanges the [B] column sums with the other ranks through
 * peer-mapped mailboxes (no host-launched collective per iteration), and returns the gradient rows of its
 * own samples.  Collectives left to the caller, once per evaluation: MIN of `shift` [3] after
 * kccot_shard_local_min, SUM of cost_partial [3,2] (cost_n = partial[n,1] * eps / log2(e) + shift[n] *
 * partial[n,0]), all-to-all of the Cbar_xy / Cbar_yy row panels into column panels XYcol, YYcol [B,Brows],
 * SUM of the two M-gradient partials.
 *   mbox_ptrs[r] / flag_ptrs[r]: device pointers (valid on THIS device) to rank r's mailbox
 *   (kccot_shard_mailbox_bytes) and flag array (nranks x KCCOT_SHARD_FLAGS_PER_RANK x uint64, zeroed once: one flag
 *   per source rank and CTA of the persistent kernel).  epoch_base: any number larger
 *   than every epoch used so far, identical on all ranks (e.g. launch counter << 24).
 * ------------------------------------------------------------------------------------------ */
size_t kccot_shard_cost_workspace_bytes(int B, long long K, int Brows);
int kccot_shard_cost_fwd(const float* real, const float* fake, int B, long long K, int row0, int Brows,
                         const float* h_fake, const float* m_real, const float* h_real,
                         const float* m_fake, int T, int J, float s, float* C3rows, void* ws,
                         size_t ws_bytes, void* stream);
/* `ws` must be the workspace of the matching kccot_shard_cost_fwd call (it carries the transposed split). */
int kccot_shard_cost_bwd(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B, long long K,
                         int row0, int Brows, const float* h_fake, const float* m_real,
                         const float* h_real, const float* m_fake, int T, int J, float s,
                         float* g_fake_rows, float* gh_fake_rows, float* gm_real_part,
                         float* gh_real_rows, float* gm_fake_part, void* ws, size_t ws_bytes, void* stream);
/* bf16 videos — the row-sharded cost for callers that keep their videos in bf16.  real / fake and g_fake_rows are
 * raw bf16 bits (uint16_t), 16-byte aligned; everything else, including the workspace
 * (kccot_shard_cost_workspace_bytes), is as in the fp32 entries above, and g_fake_rows may be NULL.
 * Contract: the results are EXACTLY those of the fp32 entries on the widened videos (a bf16 value is exact in fp32):
 * C3rows and the h / M gradients bit for bit, g_fake_rows the fp32 gradient rows rounded to nearest even.  The
 * pre-pass widens on load and runs the fp32 instruction sequence; the adjoint GEMM rounds only at its store.  No fp32
 * copy of a video is made.  Null pointers, a bad row range and a video or gradient pointer that is not 16-byte
 * aligned are rejected (KCCOT_EINVAL) before any CUDA call.  The Sinkhorn entries below see only fp32 cost rows. */
int kccot_shard_cost_fwd_bf16(const uint16_t* real, const uint16_t* fake, int B, long long K, int row0,
                              int Brows, const float* h_fake, const float* m_real, const float* h_real,
                              const float* m_fake, int T, int J, float s, float* C3rows, void* ws,
                              size_t ws_bytes, void* stream);
int kccot_shard_cost_bwd_bf16(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B,
                              long long K, int row0, int Brows, const float* h_fake, const float* m_real,
                              const float* h_real, const float* m_fake, int T, int J, float s,
                              uint16_t* g_fake_rows, float* gh_fake_rows, float* gm_real_part,
                              float* gh_real_rows, float* gm_fake_part, void* ws, size_t ws_bytes,
                              void* stream);
/* Shared context frames in the row shards — the hint of kccot_mixed_loss_fwd_ctx for the sharded cost: every column c
 * of the flattened [B, K] rows with (c % ctx_period) < ctx_len holds identical values in real and fake (for
 * [B,H,T,W,C] videos ctx_period = T*W*C, ctx_len = ctx_frames*W*C).  Arguments as in the plain / _bf16 entries above,
 * plus the hint; the workspace is kccot_shard_cost_workspace_bytes_ctx (0 for a bad hint), and the backward needs the
 * workspace of the matching forward call with the same hint.
 *   fwd: fake's context columns are never read; where a fake row's context value is needed (column statistics, row
 *        norms) the real row's value stands in.  The Gram of the context columns is computed once (this rank's real
 *        rows x all reals) and shared by the xy, xx and yy blocks, which add the Gram of the predicted columns to it.
 *   results: equal to the plain entries' on inputs that keep the promise, within floating-point tolerance: not bit
 *        for bit, because the context and predicted parts of each dot product are summed separately.
 *   bwd: g_fake_rows is the gradient with respect to the PREDICTED columns; its context columns are written as zero
 *        (as kccot_mixed_loss_bwd_ctx does).  The h / M gradients are those of the plain entry on the same cost
 *        adjoints.  The _bf16_ctx twins keep the bf16 contract: the results of the fp32 _ctx entries on the widened
 *        videos, g_fake_rows rounded to nearest even.
 *   ctx_len == 0: no hint; the plain entries run, bit for bit.
 *   Rejected with KCCOT_EINVAL before any CUDA call: ctx_period < 0, ctx_len < 0, ctx_len >= ctx_period (unless both
 *   are 0), K % ctx_period != 0, K >= 2^31 - 64 with a hint, and every check of the plain / _bf16 entries, including
 *   a bad row range in the backward. */
size_t kccot_shard_cost_workspace_bytes_ctx(int B, long long K, int Brows, long long ctx_period, long long ctx_len);
int kccot_shard_cost_fwd_ctx(const float* real, const float* fake, int B, long long K, int row0, int Brows,
                             const float* h_fake, const float* m_real, const float* h_real,
                             const float* m_fake, int T, int J, float s, float* C3rows, void* ws,
                             size_t ws_bytes, void* stream, long long ctx_period, long long ctx_len);
int kccot_shard_cost_bwd_ctx(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B,
                             long long K, int row0, int Brows, const float* h_fake, const float* m_real,
                             const float* h_real, const float* m_fake, int T, int J, float s,
                             float* g_fake_rows, float* gh_fake_rows, float* gm_real_part,
                             float* gh_real_rows, float* gm_fake_part, void* ws, size_t ws_bytes,
                             void* stream, long long ctx_period, long long ctx_len);
int kccot_shard_cost_fwd_bf16_ctx(const uint16_t* real, const uint16_t* fake, int B, long long K, int row0,
                                  int Brows, const float* h_fake, const float* m_real, const float* h_real,
                                  const float* m_fake, int T, int J, float s, float* C3rows, void* ws,
                                  size_t ws_bytes, void* stream, long long ctx_period, long long ctx_len);
int kccot_shard_cost_bwd_bf16_ctx(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B,
                                  long long K, int row0, int Brows, const float* h_fake, const float* m_real,
                                  const float* h_real, const float* m_fake, int T, int J, float s,
                                  uint16_t* g_fake_rows, float* gh_fake_rows, float* gm_real_part,
                                  float* gh_real_rows, float* gm_fake_part, void* ws, size_t ws_bytes,
                                  void* stream, long long ctx_period, long long ctx_len);
size_t kccot_shard_sinkhorn_workspace_bytes(int np, int Brows, int B, int L);
size_t kccot_shard_mailbox_bytes(int np, int nranks, int B);
int kccot_shard_local_min(const float* Crows, int np, int Brows, int B, float* shift_out, void* stream);
int kccot_shard_sinkhorn_fwd(const float* Crows, int np, int Brows, int B, int row0, float eps, int L,
                             int Lmin, float thresh, int exit_on_index, float* u_hist, float* v_hist,
                             int32_t* nits, float* cost_partial, const float* shift, int nranks, int rank,
                             void* const* mbox_ptrs, void* const* flag_ptrs,
                             unsigned long long epoch_base, void* ws, size_t ws_bytes, void* stream);
int kccot_shard_sinkhorn_bwd(const float* Crows, int np, int Brows, int B, int row0, float eps, int L,
                             const float* u_hist, const float* v_hist, const int32_t* nits,
                             const float* gcost, float* Cbar_rows, const float* shift, int nranks, int rank,
                             void* const* mbox_ptrs, void* const* flag_ptrs,
                             unsigned long long epoch_base, void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Fused mixed Sinkhorn loss — gan_utils.py:204-227 (compute_sinkhorn_loss) in ONE call per direction:
 *   fwd: stacked squared distances -> three cost matrices -> three Sinkhorn solves -> 2*xy - xx - yy
 *   bwd: three reverse solves -> adjoint GEMMs -> gradients of real / fake / h_fake / m_real / h_real / m_fake
 * `saved` (kccot_mixed_loss_saved_bytes) holds what the backward needs: C3 | u_hist | v_hist | nits | cost.
 * loss [nprob]; terms [nprob,3] = (xy, xx, yy) (may be NULL).  gloss [nprob] on the device.
 * Any gradient pointer may be NULL.  eps / L are explicit here: the reference's Python entry point
 * always passes 1.0 / 100 (its eps/L arguments are swallowed, SURVEY.md §0.4).
 * ------------------------------------------------------------------------------------------ */
size_t kccot_mixed_loss_saved_bytes(int nprob, int B, int L);
size_t kccot_mixed_loss_workspace_bytes(int nprob, int B, long long K, int L);
int kccot_mixed_loss_fwd(const float* real, const float* fake, int nprob, int B, long long K,
                         const float* h_fake, const float* m_real, const float* h_real,
                         const float* m_fake, int T, int J, float s, float eps, int L, void* saved,
                         float* loss, float* terms, void* ws, size_t ws_bytes, int flags, void* stream);
int kccot_mixed_loss_bwd(const float* gloss, const float* real, const float* fake, int nprob, int B,
                         long long K, const float* h_fake, const float* m_real, const float* h_real,
                         const float* m_fake, int T, int J, float s, float eps, int L, const void* saved,
                         float* g_real, float* g_fake, float* gh_fake, float* gm_real, float* gh_real,
                         float* gm_fake, void* ws, size_t ws_bytes, int flags, void* stream);

/* Shared context frames — kernel_train.py:225-226 / :267-268 build  real = concat(real_in, real_pred) and
 * fake = concat(real_in, fake_pred)  along the time axis, so with `--kernel none` the context frames of the two
 * videos are the same numbers.  The caller states that with (ctx_period, ctx_len): every column c of the flattened
 * [B, K] rows with (c % ctx_period) < ctx_len holds identical values in real and fake.  For [B,H,T,W,C] videos
 * ctx_period = T*W*C and ctx_len = ctx_frames*W*C.
 *   fwd: fake's context columns are never read (the real rows stand in for them): results are bit-identical to
 *        kccot_mixed_loss_fwd on inputs that keep the promise.
 *   bwd: g_fake is the gradient with respect to the PREDICTED columns only; its context columns (constants of the
 *        caller: copies of the data) are not read and not computed; they are set to ZERO (left untouched under
 *        KCCOT_FLAG_ACCUMULATE).
 * The tcgen05 path skips the columns when ctx_period and ctx_len are multiples of 32 and K is a multiple of
 * ctx_period; every other path computes the plain result first, so the outcome is the same on all paths.
 * Not valid after temporal / 3-D smoothing (which leaks predicted frames into context frames). */
int kccot_mixed_loss_fwd_ctx(const float* real, const float* fake, int nprob, int B, long long K,
                             const float* h_fake, const float* m_real, const float* h_real,
                             const float* m_fake, int T, int J, float s, float eps, int L, void* saved,
                             float* loss, float* terms, void* ws, size_t ws_bytes, int flags, void* stream,
                             long long ctx_period, long long ctx_len);
int kccot_mixed_loss_bwd_ctx(const float* gloss, const float* real, const float* fake, int nprob, int B,
                             long long K, const float* h_fake, const float* m_real, const float* h_real,
                             const float* m_fake, int T, int J, float s, float eps, int L, const void* saved,
                             float* g_real, float* g_fake, float* gh_fake, float* gm_real, float* gh_real,
                             float* gm_fake, void* ws, size_t ws_bytes, int flags, void* stream,
                             long long ctx_period, long long ctx_len);

/* bf16 videos — the mixed loss for callers that keep their videos in bf16 (e.g. under bf16 autocast).
 * real / fake and g_real / g_fake are raw bf16 bits (uint16_t), 16-byte aligned; h, M, their gradients, `saved`,
 * loss, terms and gloss stay fp32, and `saved` is sized by kccot_mixed_loss_saved_bytes as for fp32.  Arguments as
 * in the _ctx entries above (ctx_period = ctx_len = 0: no hint).
 * Contract: the results are EXACTLY those of the fp32 entries on the widened videos (a bf16 value is exact in fp32):
 * loss, terms and the h / M gradients bit for bit, g_real / g_fake the fp32 gradient rounded to nearest even.
 * Paths: with B <= 64, B % 8 == 0, K % 8 == 0, K >= 128 and a path flag other than KCCOT_PATH_SIMT the tcgen05
 * kernels read and write bf16 directly (no fp32 copy; the workspace is that of the fp32 call).  Every other shape
 * widens the videos into the workspace, runs the fp32 chain and rounds the gradients.
 * KCCOT_FLAG_ACCUMULATE is rejected (KCCOT_EINVAL): accumulating in bf16 would round at every call.  So is a video
 * or gradient pointer that is not 16-byte aligned. */
size_t kccot_mixed_loss_workspace_bytes_bf16(int nprob, int B, long long K, int L, int flags);
int kccot_mixed_loss_fwd_bf16(const uint16_t* real, const uint16_t* fake, int nprob, int B, long long K,
                              const float* h_fake, const float* m_real, const float* h_real,
                              const float* m_fake, int T, int J, float s, float eps, int L, void* saved,
                              float* loss, float* terms, void* ws, size_t ws_bytes, int flags, void* stream,
                              long long ctx_period, long long ctx_len);
int kccot_mixed_loss_bwd_bf16(const float* gloss, const uint16_t* real, const uint16_t* fake, int nprob,
                              int B, long long K, const float* h_fake, const float* m_real,
                              const float* h_real, const float* m_fake, int T, int J, float s, float eps,
                              int L, const void* saved, uint16_t* g_real, uint16_t* g_fake, float* gh_fake,
                              float* gm_real, float* gh_real, float* gm_fake, void* ws, size_t ws_bytes,
                              int flags, void* stream, long long ctx_period, long long ctx_len);

/* ------------------------------------------------------------------------------------------
 * Martingale penalty p_M — gan_utils.py:179-201.  M [B,T,J]; pm [1]; gM [B,T,J] = gpm * dpm/dM.
 * ------------------------------------------------------------------------------------------ */
int kccot_pm_fwd(const float* M, int B, int T, int J, float reg_lam, float s, float* pm,
                 float* stats /* [2*J + (T-1)*J] saved: mean_j, std_j, A_tj */, void* stream);
int kccot_pm_bwd(const float* M, int B, int T, int J, float reg_lam, float s, const float* stats,
                 const float* gpm /* device scalar */, float* gM, void* stream);

/* Batched independent problems — nprob penalties in one call per direction (config 4's discriminator step: one p_M per
 * problem; folding the problems into the batch axis would give one penalty over all of them, since the mean, sigma_j
 * and A_tj are taken over the batch).  M [nprob,B,T,J] contiguous; pm [nprob]; stats [nprob, 2*J + (T-1)*J]
 * (caller-owned, written by the forward, read by the backward; row p as in kccot_pm_fwd); gpm [nprob] on the device;
 * gM [nprob,B,T,J].  The forward runs one CTA per problem, the backward one thread per element of the batch.
 * Contract, for each problem p against kccot_pm_fwd / _bwd called on M[p] with upstream gradient gpm[p]: pm[p], stats
 * row p and gM[p] are bit-identical (both sides run the same instructions in the same order).  A problem whose M is
 * constant along some j (sigma_j = 0) takes the single call's sigma_j = 0 branch and changes no other problem's numbers.
 * The argument checks are the single entries' (null pointers, B >= 1, T >= 2, J >= 1, and in the forward the
 * shared-memory cap on T*J) plus 1 <= nprob <= 65535, all KCCOT_EINVAL and all made before any CUDA call.  Both calls
 * only enqueue work (no allocation, no host synchronisation) and are graph-capturable. */
int kccot_pm_batched_fwd(const float* M, int nprob, int B, int T, int J, float reg_lam, float s, float* pm,
                         float* stats, void* stream);
int kccot_pm_batched_bwd(const float* M, int nprob, int B, int T, int J, float reg_lam, float s, const float* stats,
                         const float* gpm, float* gM, void* stream);

/* ------------------------------------------------------------------------------------------
 * Gaussian kernel smoothing — data_utils.py:503-521 (temporal_convolution, mode 1) and
 * :552-582 (gaussian_convolution3D, mode 3).  x, out [B,H,T,W,C].  out = conv(x) / max(conv(x)) with REFLECT
 * padding; maxval [1] is saved for the backward.
 * taps_t / taps_s are HOST arrays of 2*radius+1 normalised weights (gaussian_kernel1d, data_utils.py:483-491);
 * they travel as kernel arguments: no filter matrix in device memory and no copy when sigma is annealed every
 * step (:584-586).  Mode 1 filters T with (taps_t, radius_t); mode 3 filters H, T and W with (taps_s, radius_s)
 * (the reference's 3-D kernel uses the spatial size for all three axes, :553,562-564).  radius 1..6, axes up to
 * 1024 and longer than the radius.
 * ------------------------------------------------------------------------------------------ */
size_t kccot_smooth_workspace_bytes(int mode, int B, int H, int T, int W, int C);
int kccot_smooth_fwd(int mode, const float* x, int B, int H, int T, int W, int C, const float* taps_t,
                     int radius_t, const float* taps_s, int radius_s, float* out, float* maxval, void* ws,
                     size_t ws_bytes, void* stream);
int kccot_smooth_bwd(int mode, const float* gout, const float* out, const float* maxval, int B, int H,
                     int T, int W, int C, const float* taps_t, int radius_t, const float* taps_s,
                     int radius_s, float* gx, void* ws, size_t ws_bytes, void* stream);

/* bf16 videos — the smoothing for callers that keep their videos in bf16.  x, out, gout and gx are raw bf16 bits
 * (uint16_t), any alignment; maxval, the taps and the workspace (kccot_smooth_workspace_bytes: mode 3 keeps its two
 * intermediates in fp32) are as in the fp32 entries, and so are the argument checks, error codes and limits.
 * `ties` [kccot_smooth_ties_bytes] is a caller-owned bit mask, 4-byte aligned, written by the forward (which zeroes it
 * first) and read by the backward: bit e % 32 of word e / 32 is set where element e is a tied maximum.
 * Contract, for bf16 x (a bf16 value is exact in fp32):
 *   fwd: out is kccot_smooth_fwd on the widened x rounded to nearest even, maxval bit-identical.  The kernels widen on
 *        load, keep every intermediate in fp32 with the fp32 coefficients and FMA order, and round only at the store.
 *   ties: the elements whose fp32 quotient conv(x) / maxval is exactly 1.0f, the set the fp32 backward finds with
 *        out == 1.0f.  The bf16 out cannot carry it: every fp32 value in [1 - 2^-9, 1) rounds to 1.0.
 *   bwd: gx is the fp32 backward on the widened gout rounded to nearest even, bit for bit at every element outside
 *        the adjoint stencil's support of the tied maxima; inside it gx differs only through S = sum(gout * out),
 *        which is formed from the bf16 out.  The tie count is the popcount of the mask.
 * Both calls are graph-capturable (the taps travel as kernel arguments; the mask and the sums are cleared with
 * cudaMemsetAsync). */
size_t kccot_smooth_ties_bytes(int B, int H, int T, int W, int C);   /* ceil(B*H*T*W*C / 32) * 4 */
int kccot_smooth_fwd_bf16(int mode, const uint16_t* x, int B, int H, int T, int W, int C,
                          const float* taps_t, int radius_t, const float* taps_s, int radius_s,
                          uint16_t* out, float* maxval, uint32_t* ties, void* ws, size_t ws_bytes,
                          void* stream);
int kccot_smooth_bwd_bf16(int mode, const uint16_t* gout, const uint16_t* out, const float* maxval,
                          const uint32_t* ties, int B, int H, int T, int W, int C, const float* taps_t,
                          int radius_t, const float* taps_s, int radius_s, uint16_t* gx, void* ws,
                          size_t ws_bytes, void* stream);

/* Weights in device memory — the smoothing for a sigma that changes between replays of a captured CUDA graph (an
 * annealed sigma, :584-586), which host weights cannot follow: a graph records kernel arguments once.  Each entry has
 * the arguments of its twin above, except that the two host arrays (taps_t, radius_t, taps_s, radius_s) become one
 * device array `taps_dev` of 2*radius+1 fp32 weights, 4-byte aligned, and its radius: mode 1 filters T with them,
 * mode 3 filters H, T and W with them.  The kernels read taps_dev when they run, so it may be rewritten between
 * replays; it must hold its values until the call's kernels have run.
 * Contract, for the same weight values: out, maxval and the tie mask are bit-identical to the twin's; gx is
 * bit-identical outside the adjoint stencil of the tied maxima, where S = sum(gout * out) is an order-dependent atomic
 * sum in both.  The argument checks are the twin's (the backward entries also check the sizes, as the bf16 ones do)
 * plus a null or misaligned taps_dev (KCCOT_EINVAL), all made before any CUDA call, with the twin's error codes. */
int kccot_smooth_fwd_dev(int mode, const float* x, int B, int H, int T, int W, int C, const float* taps_dev,
                         int radius, float* out, float* maxval, void* ws, size_t ws_bytes, void* stream);
int kccot_smooth_bwd_dev(int mode, const float* gout, const float* out, const float* maxval, int B, int H,
                         int T, int W, int C, const float* taps_dev, int radius, float* gx, void* ws,
                         size_t ws_bytes, void* stream);
int kccot_smooth_fwd_bf16_dev(int mode, const uint16_t* x, int B, int H, int T, int W, int C,
                              const float* taps_dev, int radius, uint16_t* out, float* maxval, uint32_t* ties,
                              void* ws, size_t ws_bytes, void* stream);
int kccot_smooth_bwd_bf16_dev(int mode, const uint16_t* gout, const uint16_t* out, const float* maxval,
                              const uint32_t* ties, int B, int H, int T, int W, int C, const float* taps_dev,
                              int radius, uint16_t* gx, void* ws, size_t ws_bytes, void* stream);

/* Batched independent problems — nprob videos [B,H,T,W,C] that lie contiguously as [nprob,B,H,T,W,C] (x, out, gout,
 * gx), smoothed in one call: problem p is filtered with its own weights, row p of `taps_dev` [nprob, 2*radius+1] (fp32,
 * device memory, 4-byte aligned, read when the kernels run, as in the *_dev entries), and divided by its own maximum,
 * maxval[p] [nprob], which the forward writes and the backward reads.  Mode 1 filters T, mode 3 filters H, T and W.
 * The workspace (kccot_smooth_batched_workspace_bytes, 16-byte aligned) holds 2*nprob tie sums, and in mode 3 two fp32
 * intermediates of nprob*B*H*T*W*C floats; the forward needs it in mode 3 only, the backward always.  The _bf16 twins
 * take bf16 x / out / gout / gx (raw bits, any alignment) and one caller-owned tie mask over the whole batch,
 * kccot_smooth_ties_bytes(nprob*B, H, T, W, C) bytes, 4-byte aligned: bit (p*n + e) % 32 of word (p*n + e) / 32 marks
 * element e of problem p (n = B*H*T*W*C), so a word may hold bits of two problems.  The forward zeroes it first.
 * Contract, for each problem p against the *_dev twin called on problem p's video with weights row p: out[p], maxval[p]
 * and the tie-mask bits of problem p are bit-identical; gx[p] is bit-identical outside the adjoint stencil of p's
 * tied maxima, where both sides form S_p = sum(gout * out) with atomics in a run-dependent order.  A tie in one problem
 * changes no other problem's numbers.  The argument checks are the twin's plus 1 <= nprob <= 65535 (KCCOT_EINVAL), all
 * made before any CUDA call, with the twin's error codes.  Both calls are graph-capturable. */
size_t kccot_smooth_batched_workspace_bytes(int mode, int nprob, int B, int H, int T, int W, int C);
int kccot_smooth_batched_fwd(int mode, const float* x, int nprob, int B, int H, int T, int W, int C,
                             const float* taps_dev, int radius, float* out, float* maxval, void* ws,
                             size_t ws_bytes, void* stream);
int kccot_smooth_batched_bwd(int mode, const float* gout, const float* out, const float* maxval, int nprob, int B,
                             int H, int T, int W, int C, const float* taps_dev, int radius, float* gx, void* ws,
                             size_t ws_bytes, void* stream);
int kccot_smooth_batched_fwd_bf16(int mode, const uint16_t* x, int nprob, int B, int H, int T, int W, int C,
                                  const float* taps_dev, int radius, uint16_t* out, float* maxval, uint32_t* ties,
                                  void* ws, size_t ws_bytes, void* stream);
int kccot_smooth_batched_bwd_bf16(int mode, const uint16_t* gout, const uint16_t* out, const float* maxval,
                                  const uint32_t* ties, int nprob, int B, int H, int T, int W, int C,
                                  const float* taps_dev, int radius, uint16_t* gx, void* ws, size_t ws_bytes,
                                  void* stream);

#ifdef __cplusplus
}
#endif
#endif /* KCCOT_H_ */
