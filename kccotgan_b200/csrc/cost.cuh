// Internal interfaces of the cost path (shared by cost_simt.cu, gram_tcgen05.cu, cost_abi.cu).
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"

namespace kccot {

// One cost matrix to finalise: C[p,i,j] = s * sum_ks part[...] + s * martingale terms.
struct CostBlock {
  const float* part;       // partial squared distances
  long long prob_stride;   // elements between problems in `part`
  long long ks_stride;     // elements between k-slabs
  int ld, row_off, col_off, nks;
  const float *h1, *M1, *h2, *M2;   // martingale pairs (row-indexed h, column-indexed M); may be null
  float* C;
  long long C_prob_stride;
  int Bx, By, zero_diag;
  int sym;                 // partials hold only hi.lo^T of the cross terms: C_ij = (P_ij + P_ji) / 2 (tensor-core path)
  int tiled;               // tensor-core partial layout part[p][16 x 16 tiles of 8 x 8][ks][64] (sym implied)
};
struct CostBlocks {
  CostBlock b[3];
  int* zero = nullptr;     // optional [nprob] counters cleared by the finalize kernel (see SinkhornMix)
};

// One output tensor of the martingale adjoint (see martingale_bwd_kernel).
struct MartJob {
  float* out;                 // [nprob, nrows, T, J]; null = skip
  const float *C1, *X1;       // first product: weights from Cbar matrix C1, factors from X1 [nprob, ncontr, T, J]
  const float *C2, *X2;       // optional second product
  long long cprob;            // elements between problems in C1 / C2
  int ld, nrows, ncontr;      // Cbar leading dimension; output rows; contraction length
  int transposed;             // 0: W[r,k] = C[r*ld + k];  1: W[r,k] = C[k*ld + r]
  int mode;                   // 0: factors are first differences of M;  1: shifted differences of h
  int acc;                    // add into `out`
};
struct MartJobs {
  MartJob j[4];
};
int launch_martingale_jobs(const MartJobs& jobs, int njobs, int nprob, int T, int J, float s, cudaStream_t st);

// cost_simt.cu
void choose_ksplit_simt(int nprob, int Bx, int By, long long K, int* ksplit, long long* kslab);
int launch_sqdist_partials_simt(const float* x, const float* y, int nprob, int Bx, int By, long long K,
                                int ksplit, long long kslab, float* part, cudaStream_t st);
// kccot_mixed_cost_fwd plus optional counters for the finalize kernel to clear (mixed_abi.cu)
int mixed_cost_fwd_impl(const float* real, const float* fake, int nprob, int B, long long K, const float* h_fake,
                        const float* m_real, const float* h_real, const float* m_fake, int T, int J, float s,
                        float* C3, void* ws, size_t ws_bytes, int flags, void* stream, int* zero_counters);
// the tensor-core path of kccot_mixed_cost_fwd / _bwd for bf16 videos and gradients (raw bits; cost_abi.cu)
int mixed_cost_fwd_bf16_tc(const uint16_t* real, const uint16_t* fake, int nprob, int B, long long K,
                           const float* h_fake, const float* m_real, const float* h_real, const float* m_fake, int T,
                           int J, float s, float* C3, void* ws, size_t ws_bytes, cudaStream_t st, int* zero_counters);
int mixed_cost_bwd_bf16_tc(const float* Cbar3, const uint16_t* real, const uint16_t* fake, int nprob, int B,
                           long long K, const float* h_fake, const float* m_real, const float* h_real,
                           const float* m_fake, int T, int J, float s, uint16_t* g_real, uint16_t* g_fake,
                           float* gh_fake, float* gm_real, float* gh_real, float* gm_fake, void* ws, size_t ws_bytes,
                           cudaStream_t st);
int launch_cost_finalize(const CostBlocks& blocks, int nblocks, int nprob, int T, int J, float s,
                         cudaStream_t st);
int launch_cost_bwd_simt(const float* W, long long sr, long long sc, long long wprob, const float* a,
                         const float* b, int nprob, int Ba, int Bb, long long K, float s, float* g,
                         int accumulate, cudaStream_t st);
int launch_martingale_bwd(const float* Cbar, long long cprob, const float* h, const float* M, int nprob,
                          int Bx, int By, int T, int J, float s, float w, float* gh, float* gM,
                          int acc_h, int acc_M, cudaStream_t st);

// gram_tcgen05.cu — stacked-row tensor-core path.  Z = [x; y] (or x alone when y == nullptr),
// R = rows of Z <= 128.  Writes partial squared-distance tiles part[p][ks][128][128].
bool tc_sqdist_supported(const float* x, const float* y, int Bx, int By, long long K);
void tc_sqdist_plan(int nprob, int R, long long K, int* ksplit, int* kblocks_per_slab);
int launch_sqdist_partials_tc(const float* x, const float* y, int nprob, int Bx, int By, long long K,
                              int ksplit, int kblocks_per_slab, float* part, cudaStream_t st);
// bf16 videos (raw bits, K % 8 == 0, 16-byte aligned): the same partials as the fp32 launcher on widened copies
bool tc_sqdist_bf16_supported(int Bx, int By, long long K);
int launch_sqdist_partials_tc_bf16(const uint16_t* x, const uint16_t* y, int nprob, int Bx, int By, long long K,
                                   int ksplit, int kblocks_per_slab, float* part, cudaStream_t st);

// grad_tcgen05.cu — tensor-core adjoint over the stacked rows z = [x; y] (see the file header).
// Wws: tc_grad_ws_bytes(nprob) of scratch for the W' images.  gx / gy may be null.
bool tc_grad_supported(const float* x, const float* y, int Bx, int By, long long K, const float* gx,
                       const float* gy);
size_t tc_grad_ws_bytes(int nprob);      // scratch of the two launchers below (W' images)
int launch_grad_tc(const float* Cbar3, const float* x, const float* y, int nprob, int Bx, int By, long long K,
                   float s, float* gx, float* gy, int accumulate, float* Wws, cudaStream_t st);
// bf16 videos and gradients of the mixed loss (B <= 64, K % 8 == 0, 16-byte aligned): gx / gy equal the fp32
// launcher's result on the widened videos rounded to nearest even; no accumulation
int launch_grad_tc_bf16(const float* Cbar3, const uint16_t* x, const uint16_t* y, int nprob, int B, long long K,
                        float s, uint16_t* gx, uint16_t* gy, float* Wws, cudaStream_t st);
int launch_grad_pair_tc(const float* Cbar, const float* x, const float* y, int nprob, int Bx, int By, long long K,
                        float s, float* gx, float* gy, int accumulate, float* Wws, cudaStream_t st);

// ------------------------------------------------------------------------------------------------
// Large-batch path (B > 64): gemm_f16x3.cu / large_prep.cu / large_abi.cu
// ------------------------------------------------------------------------------------------------
#define G3_BN 256        // square output tile of gemm_f16x3.cu (large_prep.cu reads it for the symmetric blocks)
#define G3_BK 64
struct G3Job {
  int a_row0, b_row0;      // first row of this block in the A / B operand arrays
  int m, n;                // valid rows / columns of the block
  int tm, tn, ntiles;      // filled by g3_count_tiles_pair
  int tri;                 // symmetric block (a_row0 == b_row0): only tiles touching the upper triangle
  float* out;              // [ksplit][m][ld] (bf16 bits for launch_gemm_f16x3_pair_bf16)
  long long ld, ks_stride;
};
struct G3Params {
  G3Job job[3];
  int njobs, ntiles_total;
  int nkb, ksplit, kb_per_split;
  int drain;               // k-blocks per accumulation chunk (see gemm_f16x3.cu)
  float alpha;
  const float* alpha_dev;  // optional device scalar multiplied into alpha
  int accumulate;          // add into `out` instead of overwriting it
};
int g3_count_tiles_pair(G3Job* jb);     // 256 x 256 tiles of the CTA-pair kernel
// `units`: clusters to fill
void g3_plan_split(int ntiles, int nkb, int units, int* ksplit, int* kb_per_split);
// A*: [a_rows][a_pitch] fp16 (hi, lo), B*: [b_rows][b_pitch]; contraction over `kdim` leading columns
int launch_gemm_f16x3_pair(const __half* A1, const __half* A2, long long a_rows, long long a_pitch_elems,
                           const __half* B1, const __half* B2, long long b_rows, long long b_pitch_elems, long long kdim,
                           G3Params P, cudaStream_t st);
// the same product stored as bf16 (the fp32 output value rounded to nearest even); P.accumulate must be 0
int launch_gemm_f16x3_pair_bf16(const __half* A1, const __half* A2, long long a_rows, long long a_pitch_elems,
                                const __half* B1, const __half* B2, long long b_rows, long long b_pitch_elems,
                                long long kdim, G3Params P, cudaStream_t st);

// large_abi.cu: true when the large-batch path takes the shape
bool large_path_wanted(int Bx, int By, bool same);
size_t large_cost_fwd_ws_bytes(int Bx, int By, long long K, bool same, bool mixed);
size_t large_cost_bwd_ws_bytes(int Bx, int By, long long K, bool mixed);
int large_mixed_cost_fwd(const float* real, const float* fake, int B, long long K, const float* h_fake,
                         const float* m_real, const float* h_real, const float* m_fake, int T, int J, float s,
                         float* C3, void* ws, size_t ws_bytes, cudaStream_t st);
int large_mixed_cost_bwd(const float* Cbar3, const float* real, const float* fake, int B, long long K, float s,
                         float* g_real, float* g_fake, int accumulate, void* ws, size_t ws_bytes, cudaStream_t st);
int large_cost_fwd(const float* x, const float* y, int Bx, int By, long long K, const float* h1, const float* M1,
                   const float* h2, const float* M2, int T, int J, float s, float* C, void* ws, size_t ws_bytes,
                   cudaStream_t st);
int large_cost_bwd(const float* Cbar, const float* x, const float* y, int Bx, int By, long long K, float s, float* gx,
                   float* gy, int accumulate, void* ws, size_t ws_bytes, cudaStream_t st);
size_t large_shard_ws_bytes(int B, long long K, int Brows);
int large_shard_cost_fwd(const float* real, const float* fake, int B, long long K, int row0, int Brows, const float* h_fake,
                         const float* m_real, const float* h_real, const float* m_fake, int T, int J, float s,
                         float* C3rows, void* ws, size_t ws_bytes, cudaStream_t st);
int large_shard_cost_bwd(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B, long long K, int row0,
                         int Brows, const float* h_fake, const float* m_real, const float* h_real, const float* m_fake,
                         int T, int J, float s, float* g_fake_rows, float* gh_fake_rows, float* gm_real_part,
                         float* gh_real_rows, float* gm_fake_part, void* ws, size_t ws_bytes, cudaStream_t st);
// bf16 videos and fake gradient rows (raw bits): the fp32 results on the widened videos, the gradient rows rounded to
// nearest even; same workspace
int large_shard_cost_fwd(const uint16_t* real, const uint16_t* fake, int B, long long K, int row0, int Brows,
                         const float* h_fake, const float* m_real, const float* h_real, const float* m_fake, int T, int J,
                         float s, float* C3rows, void* ws, size_t ws_bytes, cudaStream_t st);
int large_shard_cost_bwd(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B, long long K, int row0,
                         int Brows, const float* h_fake, const float* m_real, const float* h_real, const float* m_fake,
                         int T, int J, float s, uint16_t* g_fake_rows, float* gh_fake_rows, float* gm_real_part,
                         float* gh_real_rows, float* gm_fake_part, void* ws, size_t ws_bytes, cudaStream_t st);
// shared context frames (kccot_shard_cost_*_ctx; the caller has checked K < 2^31 - 64, K % period == 0 and
// 0 < clen < period): fake's context columns are not read, g_fake_rows' context columns are written as zero.  Own
// workspace size; the backward needs the workspace of the matching forward.
size_t large_shard_ws_bytes_ctx(int B, long long K, int Brows, long long period, long long clen);
int large_shard_cost_fwd_ctx(const float* real, const float* fake, int B, long long K, int row0, int Brows,
                             const float* h_fake, const float* m_real, const float* h_real, const float* m_fake, int T,
                             int J, float s, float* C3rows, void* ws, size_t ws_bytes, long long period, long long clen,
                             cudaStream_t st);
int large_shard_cost_fwd_ctx(const uint16_t* real, const uint16_t* fake, int B, long long K, int row0, int Brows,
                             const float* h_fake, const float* m_real, const float* h_real, const float* m_fake, int T,
                             int J, float s, float* C3rows, void* ws, size_t ws_bytes, long long period, long long clen,
                             cudaStream_t st);
int large_shard_cost_bwd_ctx(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B, long long K, int row0,
                             int Brows, const float* h_fake, const float* m_real, const float* h_real,
                             const float* m_fake, int T, int J, float s, float* g_fake_rows, float* gh_fake_rows,
                             float* gm_real_part, float* gh_real_rows, float* gm_fake_part, void* ws, size_t ws_bytes,
                             long long period, long long clen, cudaStream_t st);
int large_shard_cost_bwd_ctx(const float* Cbar3rows, const float* XYcol, const float* YYcol, int B, long long K, int row0,
                             int Brows, const float* h_fake, const float* m_real, const float* h_real,
                             const float* m_fake, int T, int J, float s, uint16_t* g_fake_rows, float* gh_fake_rows,
                             float* gm_real_part, float* gh_real_rows, float* gm_fake_part, void* ws, size_t ws_bytes,
                             long long period, long long clen, cudaStream_t st);

}  // namespace kccot
