// Internal interfaces of the large-batch cost path (large_prep.cu, large_abi.cu).
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"

namespace kccot {

// device scalars shared by the passes of one call (floats / raw bits), zeroed by large_launch_stats
enum {
  kScalAbsmax = 0,     // bits of max |z| over the stacked rows
  kScalZscale = 1,     // 2^e applied to the centred rows before the fp16 split
  kScalZinv = 2,       // 2^-e
  kScalWabs = 3,       // bits of max |W_rc|, r != c
  kScalDabs = 4,       // bits of max |rowsum W|
  kScalGradAlpha = 5,  // 1 / (W' scale * z scale): multiplied into the adjoint GEMM's alpha
  kScalCount = 8
};

struct LargeFinBlock {
  const float* P;            // raw dot products [nks][.][ld]
  long long ld, ks_stride;
  int nks, tri;
  const float *ni, *nj;      // row norms of the block's row / column samples
  const float *h1, *M1, *h2, *M2;
  float* C;
  long long ldc;
  int Bx, By, zero_diag;
  int diag_off;              // the self-distance zero sits at j == i + diag_off (row shards: the block's first global row)
};
struct LargeFin {
  LargeFinBlock b[3];
};

int large_launch_stats(const float* x, const float* y, int Bx, int By, long long K, int nseg, float* part, float* mean,
                       float* scal, cudaStream_t st);
int large_launch_split(const float* x, const float* y, int Bx, int By, long long K, long long Kp, int Rp,
                       const float* mean, const float* scal, __half* Zh1, __half* Zh2, __half* ZT1, __half* ZT2,
                       cudaStream_t st);
// bf16 videos (raw bits): the same column sums, scale and split as the fp32 launchers on the widened videos
int large_launch_stats(const uint16_t* x, const uint16_t* y, int Bx, int By, long long K, int nseg, float* part,
                       float* mean, float* scal, cudaStream_t st);
int large_launch_split(const uint16_t* x, const uint16_t* y, int Bx, int By, long long K, long long Kp, int Rp,
                       const float* mean, const float* scal, __half* Zh1, __half* Zh2, __half* ZT1, __half* ZT2,
                       cudaStream_t st);
// Shared context frames of the row shards (B real rows x, B fake rows y; K < 2^31, K % period == 0,
// 0 < clen < period): column c is a context column when c % period < clen, and y's values there are never read (x's
// stand in).  The stats are those of large_launch_stats on inputs that keep that promise.  The split writes the columns
// permuted: the nc = K / period * clen context columns in [0, Kcp), the predicted ones from Kcp on, each part
// zero-padded to a multiple of 64; Zh [2B][Kpp], ZT [Kpp][Rp].  The scatter writes g_pred [nrows][nq] (the predicted
// columns in order) back to the video columns of g [nrows][K] and zeroes the context columns.
int large_launch_stats_ctx(const float* x, const float* y, int B, long long K, int period, int clen, int nseg,
                           float* part, float* mean, float* scal, cudaStream_t st);
int large_launch_stats_ctx(const uint16_t* x, const uint16_t* y, int B, long long K, int period, int clen, int nseg,
                           float* part, float* mean, float* scal, cudaStream_t st);
int large_launch_split_ctx(const float* x, const float* y, int B, long long K, int period, int clen, int Kcp,
                           long long Kpp, int Rp, const float* mean, const float* scal, __half* Zh1, __half* Zh2,
                           __half* ZT1, __half* ZT2, cudaStream_t st);
int large_launch_split_ctx(const uint16_t* x, const uint16_t* y, int B, long long K, int period, int clen, int Kcp,
                           long long Kpp, int Rp, const float* mean, const float* scal, __half* Zh1, __half* Zh2,
                           __half* ZT1, __half* ZT2, cudaStream_t st);
int large_launch_ctx_scatter(const float* g_pred, int nrows, int K, int period, int clen, float* g, cudaStream_t st);
int large_launch_ctx_scatter(const uint16_t* g_pred, int nrows, int K, int period, int clen, uint16_t* g,
                             cudaStream_t st);
int large_launch_rownorm(const __half* Zh1, const __half* Zh2, int R, long long K, long long Kp, float* norms,
                         cudaStream_t st);
int large_launch_finalize(const LargeFin& F, int nblocks, int T, int J, float s, const float* scal, cudaStream_t st);
int large_launch_wbuild(const float* Cxx, const float* Cxy, const float* Cyy, int Bx, int By, int row_off, int nrows,
                        int Rp, float* Wtmp, float* rs_part, float* rowsum, float* scal, __half* Wh1, __half* Wh2,
                        cudaStream_t st);
// row shard: W' rows of the fake samples [row0, row0 + nloc) from the column panels XYcol [Bx][nloc] = Cbar_xy[:, rows],
// YYcol [By][nloc] = Cbar_yy[:, rows] (received from the other ranks) and the own rows YYrow [nloc][By] = Cbar_yy[rows, :]
int large_launch_wbuild_shard(const float* XYcol, const float* YYcol, const float* YYrow, int Bx, int By, int row0, int nloc,
                              int Rp, float* Wtmp, float* rs_part, float* rowsum, float* scal, __half* Wh1, __half* Wh2,
                              cudaStream_t st);

}  // namespace kccot
