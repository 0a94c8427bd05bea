// Tiled tensor-core GEMM of the large-batch cost path (B > 64: BASELINE config 5, B = 8192):
//
//     out[m][n] (+)= alpha * sum_k ( A1[m,k] B1[n,k] + A1[m,k] B2[n,k] + A2[m,k] B1[n,k] )
//
// A1/B1 are the fp16 "hi" halves and A2/B2 the fp16 "lo" halves of fp32 operands split by the pre-pass
// (large_prep.cu): x = hi + lo with 11 + 11 significant bits, the same mantissa width as TF32, so the three
// products reproduce 3xTF32 accuracy at the fp16 rate (2x the tf32 rate) and half the operand bytes.  The
// forward uses it as the Gram of the centred stacked rows (gan_utils.py:14-17 in GEMM form), the backward
// as W' . Z over the transposed split (the adjoint of the same lines).
//
// tcgen05 cta_group::2: a cluster of two CTAs on one TPC computes a 256 x 256 output tile.  Each CTA holds
// 128 rows of A and HALF of the B tile (128 of its 256 rows); the tensor cores of both SMs read the other half
// from the peer's shared memory, so per CTA and k-block only 64 KB are staged (A hi/lo 2 x 16 KB + B-half
// hi/lo 2 x 16 KB: 3 stages) and the shared-memory port carries 64 B/clk of operand reads instead of the 96 a
// single-CTA 128 x 256 tile needs (that tile is shared-memory bound at ~80 % of the tensor pipe).
//
//   accums   : fp32 in tensor memory: hi.hi in columns [0,256), the two cross products in columns [256,512).
//              The cross terms are 2^-11 smaller; adding them into the large accumulator would lose them to
//              the tensor core's truncating fp32 adder.
//   roles    : warp 0 = TMA producer (both CTAs; every load signals the LEADER's full barrier:
//              cp.async.bulk.tensor...cta_group::2), warp 1 = MMA issuer (leader CTA only; commits are multicast
//              to both CTAs' barriers), warps 2-9 = drain / epilogue (each CTA drains its own tensor memory:
//              lanes = its 128 rows, 256 + 256 columns).
//   chunks   : every `drain` k-blocks the hi.hi accumulator is added (round-to-nearest fp32) into REGISTER
//              accumulators of the drain warps (128 per thread) — the tensor core's own accumulation truncates —
//              and the MMA issuer resumes as soon as the tensor-memory reads have completed.  Output is written
//              once per work item.
//   work item: (job, tile, k-split).  Up to 3 jobs share the operand tensor maps and differ in row offsets
//              (the xy, xx, yy blocks of the stacked Gram); symmetric jobs enumerate only the tiles on or above
//              the diagonal.  Tiles are ordered column-major; persistent clusters, static round-robin.
#include <cuda_fp16.h>

#include "cost.cuh"
#include "tc_common.cuh"

namespace kccot {

namespace {
constexpr int PM = G3_BN, PN = G3_BN, BK = G3_BK;          // pair tile
constexpr int kABytes = 128 * BK * 2;                      // 16 KB: this CTA's 128 rows of A
constexpr int kBBytes = 128 * BK * 2;                      // 16 KB: this CTA's half of the B tile
constexpr int kStageBytes = 2 * kABytes + 2 * kBBytes;     // 64 KB
constexpr int kStages = 3;
constexpr int kEpiWarps = 8;
constexpr int kThreads = 64 + kEpiWarps * 32;              // 320
constexpr int kTmemCols = 512;
constexpr int kAccX = 256;

struct Bars {
  uint64_t full[kStages], empty[kStages];
  uint64_t acc_full, acc_free;
  uint32_t tmem_base;
};

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(const CUtensorMap* m, uint32_t bar_cluster_addr, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(tc::smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {     // arrives on `bar` in BOTH CTAs
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   tc::smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc::smem_u32(dst_smem)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

struct Item {
  int job, m0, n0, ks;
};
__device__ __forceinline__ bool decode_item(const G3Params& P, int w, Item& it) {
  int tile = w / P.ksplit;
  it.ks = w - tile * P.ksplit;
  for (int j = 0; j < P.njobs; ++j) {
    const G3Job& jb = P.job[j];
    if (tile < jb.ntiles) {
      it.job = j;
      int tni, tmi;
      if (!jb.tri) {
        tni = tile / jb.tm;
        tmi = tile - tni * jb.tm;
      } else {                              // square tiles: column tile t needs row tiles 0 .. min(tm, t + 1) - 1
        tni = 0;
        for (;; ++tni) {
          const int cnt = min(jb.tm, tni + 1);
          if (tile < cnt) break;
          tile -= cnt;
        }
        tmi = tile;
      }
      it.m0 = tmi * PM;
      it.n0 = tni * PN;
      return true;
    }
    tile -= jb.ntiles;
  }
  return false;
}
}  // namespace

// Out = float: out (+)= alpha * acc.  Out = uint16_t: out = bf16(alpha * acc), the fp32 epilogue's value rounded to
// nearest even (G3Job::out then holds bf16 bits; no accumulation).
template <typename Out>
__global__ void __launch_bounds__(kThreads, 1)
gemm_f16x3_pair_kernel(const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmA2,
                       const __grid_constant__ CUtensorMap tmB1, const __grid_constant__ CUtensorMap tmB2,
                       const __grid_constant__ G3Params P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
  Bars& bars = *reinterpret_cast<Bars*>(base + kStages * kStageBytes);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int nitems = P.ntiles_total * P.ksplit;
  const int cluster_id = blockIdx.x >> 1, nclusters = gridDim.x >> 1;

  if (threadIdx.x == 0) {
    tc::prefetch_tmap(&tmA1);
    tc::prefetch_tmap(&tmA2);
    tc::prefetch_tmap(&tmB1);
    tc::prefetch_tmap(&tmB2);
    for (int s = 0; s < kStages; ++s) {
      tc::mbar_init(&bars.full[s], 1);                     // the leader's arrive.expect_tx (both CTAs' bytes)
      tc::mbar_init(&bars.empty[s], 1);                    // one multicast commit
    }
    tc::mbar_init(&bars.acc_full, 1);
    tc::mbar_init(&bars.acc_free, 2 * kEpiWarps);          // (leader's copy) drain warps of both CTAs
    tc::fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc_pair(&bars.tmem_base, kTmemCols);
    tmem_relinquish_pair();
  }
  tc::tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                       // barriers of both CTAs are initialised
  tc::tc_fence_after();
  const uint32_t tmem = bars.tmem_base;

  if (warp == 0) {
    // ------------------------------- TMA producer (both CTAs) ----------------------------------
    if (tc::elect_one()) {
      int stage = 0, phase = 0;
      Item it;
      for (int w = cluster_id; w < nitems; w += nclusters) {
        if (!decode_item(P, w, it)) break;
        const G3Job& jb = P.job[it.job];
        const int kb0 = it.ks * P.kb_per_split, kb1 = min(P.nkb, kb0 + P.kb_per_split);
        const int arow = jb.a_row0 + it.m0 + 128 * (int)rank, brow = jb.b_row0 + it.n0 + 128 * (int)rank;
        for (int kb = kb0; kb < kb1; ++kb) {
          tc::mbar_wait(&bars.empty[stage], phase ^ 1);
          uint8_t* sb = base + (size_t)stage * kStageBytes;
          const uint32_t full_leader = mapa_u32(tc::smem_u32(&bars.full[stage]), 0);
          if (leader) tc::mbar_arrive_expect_tx(&bars.full[stage], (uint32_t)(2 * kStageBytes));
          tma_load_2d_pair(&tmA1, full_leader, sb, kb * BK, arow);
          tma_load_2d_pair(&tmB1, full_leader, sb + 2 * kABytes, kb * BK, brow);
          tma_load_2d_pair(&tmB2, full_leader, sb + 2 * kABytes + kBBytes, kb * BK, brow);
          tma_load_2d_pair(&tmA2, full_leader, sb + kABytes, kb * BK, arow);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
      // drain the asynchronous tcgen05.commit arrivals on empty[] before the CTA may exit (see grad_tcgen05.cu)
      for (int i = 0; i < kStages; ++i) {
        tc::mbar_wait(&bars.empty[stage], phase ^ 1);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------- MMA issuer (leader CTA) -----------------------------------
    if (leader && tc::elect_one()) {
      const uint32_t idesc = tc::make_idesc_f16(PM, PN, 0, 0);
      int stage = 0, phase = 0;
      uint32_t g = 0;
      Item it;
      for (int w = cluster_id; w < nitems; w += nclusters) {
        if (!decode_item(P, w, it)) break;
        const int kb0 = it.ks * P.kb_per_split, kb1 = min(P.nkb, kb0 + P.kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          const int rel = kb - kb0;
          const bool chunk_first = (rel % P.drain) == 0;
          const bool chunk_last = ((rel + 1) % P.drain) == 0 || kb == kb1 - 1;
          if (chunk_first) {
            tc::mbar_wait(&bars.acc_free, (g & 1u) ^ 1u);
            tc::tc_fence_after();
          }
          tc::mbar_wait(&bars.full[stage], phase);
          tc::tc_fence_after();
          const uint32_t sb = tc::smem_u32(base + (size_t)stage * kStageBytes);
#pragma unroll
          for (int k4 = 0; k4 < BK / 16; ++k4) {
            const uint64_t a1 = tc::make_smem_desc_sw128(sb + k4 * 32, 16, 1024);
            const uint64_t a2 = tc::make_smem_desc_sw128(sb + kABytes + k4 * 32, 16, 1024);
            const uint64_t b1 = tc::make_smem_desc_sw128(sb + 2 * kABytes + k4 * 32, 16, 1024);
            const uint64_t b2 = tc::make_smem_desc_sw128(sb + 2 * kABytes + kBBytes + k4 * 32, 16, 1024);
            umma_f16_pair(tmem, a1, b1, idesc, (chunk_first && k4 == 0) ? 0u : 1u);
            umma_f16_pair(tmem + kAccX, a1, b2, idesc, (rel == 0 && k4 == 0) ? 0u : 1u);
            umma_f16_pair(tmem + kAccX, a2, b1, idesc, 1u);
          }
          umma_commit_pair(&bars.empty[stage]);
          if (chunk_last) {
            umma_commit_pair(&bars.acc_full);
            ++g;
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ------------------------------- drain / epilogue (both CTAs) ------------------------------
    const int ew = warp - 2;
    const int quad = warp & 3;                              // TMEM lane quadrant this warp may read
    const int half = ew >> 2;                               // columns [128 half, 128 half + 128)
    const float alpha = P.alpha * (P.alpha_dev ? *P.alpha_dev : 1.f);
    const uint32_t free_leader = mapa_u32(tc::smem_u32(&bars.acc_free), 0);
    const uint32_t trow = tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(half * 128);
    uint32_t g = 0;
    Item it;
    for (int w = cluster_id; w < nitems; w += nclusters) {
      if (!decode_item(P, w, it)) break;
      const G3Job& jb = P.job[it.job];
      const int kb0 = it.ks * P.kb_per_split, kb1 = min(P.nkb, kb0 + P.kb_per_split);
      const int nchunks = (kb1 - kb0 + P.drain - 1) / P.drain;
      const int row = it.m0 + 128 * (int)rank + quad * 32 + lane;
      const bool row_ok = row < jb.m;
      const int ncols_left = jb.n - it.n0 - half * 128;     // valid columns of this warp's half (may be <= 0)
      float racc[128];
#pragma unroll
      for (int j = 0; j < 128; ++j) racc[j] = 0.f;
      for (int c = 0; c < nchunks; ++c) {
        tc::mbar_wait(&bars.acc_full, g & 1u);
        tc::tc_fence_after();
        const bool last = c == nchunks - 1;
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
          float d0[32];
          tc::tmem_ld_32x32(trow + (uint32_t)(cc * 32), d0);
          tc::tmem_ld_wait();
          if (cc == 3 && !last) {                           // tensor memory is free again: release the MMA issuer first
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(free_leader);
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) racc[cc * 32 + j] += d0[j];
        }
        if (last) {
          // cross accumulator, then the output tile (written once per work item)
          Out* orow = reinterpret_cast<Out*>(jb.out) + (long long)it.ks * jb.ks_stride + (long long)row * jb.ld + it.n0 +
                      half * 128;
          const bool vec_ok = ((jb.ld & 3) == 0) && ((reinterpret_cast<uintptr_t>(jb.out) & (4 * sizeof(Out) - 1)) == 0) &&
                              (((long long)it.ks * jb.ks_stride & 3) == 0) && ((it.n0 & 3) == 0);
#pragma unroll
          for (int cc = 0; cc < 4; ++cc) {
            float x[32];
            tc::tmem_ld_32x32(trow + (uint32_t)(kAccX + cc * 32), x);
            tc::tmem_ld_wait();
            if (cc == 3) {
              tc::tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive_cluster(free_leader);
            }
            const int ncols = ncols_left - cc * 32;
            if constexpr (sizeof(Out) == 2) {
              if (row_ok && ncols > 0) {
                uint16_t* o = orow + cc * 32;
                if (vec_ok && ncols >= 32) {                // 8-byte stores of four values
#pragma unroll
                  for (int j = 0; j < 8; ++j) {
                    const float v0 = fmaf(alpha, racc[cc * 32 + 4 * j + 0] + x[4 * j + 0], 0.f);
                    const float v1 = fmaf(alpha, racc[cc * 32 + 4 * j + 1] + x[4 * j + 1], 0.f);
                    const float v2 = fmaf(alpha, racc[cc * 32 + 4 * j + 2] + x[4 * j + 2], 0.f);
                    const float v3 = fmaf(alpha, racc[cc * 32 + 4 * j + 3] + x[4 * j + 3], 0.f);
                    reinterpret_cast<uint2*>(o)[j] = make_uint2(pack_bf16x2(v0, v1), pack_bf16x2(v2, v3));
                  }
                } else {
#pragma unroll
                  for (int j = 0; j < 32; ++j)
                    if (j < ncols) o[j] = __bfloat16_as_ushort(__float2bfloat16_rn(alpha * (racc[cc * 32 + j] + x[j])));
                }
              }
            } else if (row_ok && ncols > 0) {
              float* o = orow + cc * 32;
              if (vec_ok && ncols >= 32) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                  if (P.accumulate) v = reinterpret_cast<const float4*>(o)[j];
                  v.x = fmaf(alpha, racc[cc * 32 + 4 * j + 0] + x[4 * j + 0], v.x);
                  v.y = fmaf(alpha, racc[cc * 32 + 4 * j + 1] + x[4 * j + 1], v.y);
                  v.z = fmaf(alpha, racc[cc * 32 + 4 * j + 2] + x[4 * j + 2], v.z);
                  v.w = fmaf(alpha, racc[cc * 32 + 4 * j + 3] + x[4 * j + 3], v.w);
                  reinterpret_cast<float4*>(o)[j] = v;
                }
              } else {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                  if (j < ncols) {
                    const float v = alpha * (racc[cc * 32 + j] + x[j]);
                    o[j] = P.accumulate ? o[j] + v : v;
                  }
              }
            }
          }
        }
        ++g;
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                       // the peer may still read this CTA's operands / barriers
  if (warp == 1) tmem_dealloc_pair(tmem, kTmemCols);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
int g3_count_tiles_pair(G3Job* jb) {
  jb->tm = (jb->m + PM - 1) / PM;
  jb->tn = (jb->n + PN - 1) / PN;
  if (!jb->tri) {
    jb->ntiles = jb->tm * jb->tn;
  } else {
    int n = 0;
    for (int t = 0; t < jb->tn; ++t) n += (jb->tm < t + 1) ? jb->tm : t + 1;
    jb->ntiles = n;
  }
  return jb->ntiles;
}

// k-split so that the `units` clusters are filled when the tile count is small (mid-size B); each split keeps
// >= 8 k-blocks
void g3_plan_split(int ntiles, int nkb, int units, int* ksplit, int* kb_per_split) {
  int ks = 1;
  if (ntiles < units) {
    ks = (units + ntiles - 1) / ntiles;
    const int maxks = nkb / 8 > 1 ? nkb / 8 : 1;
    if (ks > maxks) ks = maxks;
  }
  int per = (nkb + ks - 1) / ks;
  *ksplit = (nkb + per - 1) / per;
  *kb_per_split = per;
}

namespace {
template <typename Out>
int launch_pair(const __half* A1, const __half* A2, long long a_rows, long long a_pitch_elems, const __half* B1,
                const __half* B2, long long b_rows, long long b_pitch_elems, long long kdim, G3Params P, cudaStream_t st) {
  CUtensorMap tA1, tA2, tB1, tB2;
  if (int rc = encode_tmap_2d_f16(&tA1, A1, (uint64_t)kdim, (uint64_t)a_rows, (uint64_t)a_pitch_elems * 2, BK, 128)) return rc;
  if (int rc = encode_tmap_2d_f16(&tA2, A2, (uint64_t)kdim, (uint64_t)a_rows, (uint64_t)a_pitch_elems * 2, BK, 128)) return rc;
  if (int rc = encode_tmap_2d_f16(&tB1, B1, (uint64_t)kdim, (uint64_t)b_rows, (uint64_t)b_pitch_elems * 2, BK, 128)) return rc;
  if (int rc = encode_tmap_2d_f16(&tB2, B2, (uint64_t)kdim, (uint64_t)b_rows, (uint64_t)b_pitch_elems * 2, BK, 128)) return rc;
  P.nkb = (int)((kdim + BK - 1) / BK);
  P.ntiles_total = 0;
  for (int j = 0; j < P.njobs; ++j) P.ntiles_total += P.job[j].ntiles;
  if (P.ntiles_total == 0) return KCCOT_OK;
  if (P.drain < 1) P.drain = 8;
  const size_t smem = (size_t)kStages * kStageBytes + sizeof(Bars) + 1024;
  static size_t attr_set[kMaxDevices] = {};
  if (smem_attr_needed(attr_set, smem))
    KCCOT_CUDA(cudaFuncSetAttribute(gemm_f16x3_pair_kernel<Out>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long nitems = (long long)P.ntiles_total * P.ksplit;
  const int max_clusters = num_sms() / 2;
  const int nclusters = (int)(nitems < max_clusters ? nitems : max_clusters);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * nclusters);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  KCCOT_CUDA(cudaLaunchKernelEx(&cfg, gemm_f16x3_pair_kernel<Out>, tA1, tA2, tB1, tB2, P));
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}
}  // namespace

int launch_gemm_f16x3_pair(const __half* A1, const __half* A2, long long a_rows, long long a_pitch_elems,
                           const __half* B1, const __half* B2, long long b_rows, long long b_pitch_elems, long long kdim,
                           G3Params P, cudaStream_t st) {
  return launch_pair<float>(A1, A2, a_rows, a_pitch_elems, B1, B2, b_rows, b_pitch_elems, kdim, P, st);
}
int launch_gemm_f16x3_pair_bf16(const __half* A1, const __half* A2, long long a_rows, long long a_pitch_elems,
                                const __half* B1, const __half* B2, long long b_rows, long long b_pitch_elems,
                                long long kdim, G3Params P, cudaStream_t st) {
  KCCOT_CHECK_ARG(!P.accumulate, "bf16 GEMM output cannot accumulate");
  return launch_pair<uint16_t>(A1, A2, a_rows, a_pitch_elems, B1, B2, b_rows, b_pitch_elems, kdim, P, st);
}

}  // namespace kccot
