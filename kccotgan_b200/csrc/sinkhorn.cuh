// Internal interfaces of the Sinkhorn kernels.
#pragma once
#include "common.cuh"

namespace kccot {

constexpr int kSmallSinkhornMaxB = 64;   // register-resident single-CTA path

// Epilogue / prologue of the mixed loss folded into the small kernels (problems come in triples xy, xx, yy):
//   forward : the CTA of a triple that finishes last writes loss[p] = 2 xy - xx - yy (gan_utils.py:225) and the
//             three terms; `counter[p]` must be zero when the kernel starts (cost_finalize_kernel clears it)
//   backward: the upstream gradient of problem n is gloss[n / 3] * (n % 3 == 0 ? 2 : -1)
struct SinkhornMix {
  float* loss = nullptr;
  float* terms = nullptr;
  int* counter = nullptr;
  const float* gloss = nullptr;
};

// sinkhorn_small.cu
int launch_sinkhorn_fwd_small(const float* C, int nsolve, int B, float eps, int L, int Lmin, float thresh,
                              int exit_on_index, float* u_hist, float* v_hist, int32_t* nits, float* cost,
                              cudaStream_t st, SinkhornMix mix = SinkhornMix());
int launch_sinkhorn_bwd_small(const float* C, int nsolve, int B, float eps, int L, const float* u_hist,
                              const float* v_hist, const int32_t* nits, const float* gcost, float* Cbar,
                              const int32_t* only_if, cudaStream_t st, SinkhornMix mix = SinkhornMix());


// sinkhorn_stream.cu — any B; C streamed from L2/HBM; a kernel boundary per half-iteration pair.
size_t stream_workspace_bytes(int B);
int stream_sinkhorn_fwd(const float* C, int B, float eps, int L, int Lmin, float thresh, int exit_on_index,
                        float* u_hist, float* v_hist, int32_t* nits, float* cost, void* ws, cudaStream_t st);
int stream_sinkhorn_bwd(const float* C, int B, float eps, int L, const float* u_hist, const float* v_hist,
                        const int32_t* nits, const float* gcost, float* Cbar, void* ws, cudaStream_t st);

// sinkhorn_persist.cu — all iterations inside one cooperative kernel (64 < B <= 8192, B % 4 == 0); row shards
// exchange their column sums inside the kernel through peer-mapped mailboxes.
constexpr int kMaxShardRanks = 8;
struct ShardComm {
  int nranks, rank;
  float* mbox[kMaxShardRanks];                 // mailbox of every rank (device pointers valid on THIS device)
  unsigned long long* flags[kMaxShardRanks];   // epoch flags of every rank, [nranks][KCCOT_SHARD_FLAGS_PER_RANK] each, zero before first use
  unsigned long long epoch0;                   // fresh for every launch and larger than any epoch used before
};
bool persist_supported(int Brows, int B, int L);
size_t persist_workspace_bytes(int np, int Brows, int B, int L);
size_t persist_mailbox_floats(int np, int nranks, int B);
int persist_sinkhorn_fwd(const float* C, int np, int Brows, int B, int row0, float eps, int L, int Lmin, float thresh,
                         int exit_on_index, float* u_hist, float* v_hist, int32_t* nits, float* cost, void* ws,
                         const ShardComm* comm, const float* shift_dev, cudaStream_t st);
int persist_sinkhorn_bwd(const float* C, int np, int Brows, int B, int row0, float eps, int L, const float* u_hist,
                         const float* v_hist, const int32_t* nits, const float* gcost, float gcost_host, float* Cbar,
                         void* ws, const ShardComm* comm, const float* shift_dev, cudaStream_t st);

}  // namespace kccot
