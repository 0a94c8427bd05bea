// Pairwise squared distances on the 5th-gen tensor cores (replaces the [B,B,T,D] broadcast of
// gan_utils.py:14-17).
//
// Stacked rows Z = [x; y] (R = Bx + By <= 128) of one problem are streamed ONCE from HBM by TMA in
// 128-byte-swizzled [R x 32] fp32 k-blocks.  Split-K: one persistent CTA per (problem, k-slab).
//   TMA warp      : fills a 4-stage ring.
//   8 convert warps: per k-block subtract the column mean (squared distance is translation
//                    invariant; centring removes the cancellation between |x|^2+|y|^2 and 2x.y),
//                    accumulate the fp32 row norms, split into tf32 hi + tf32 lo in place.  Warp w
//                    owns 16-byte chunk w of all 128 rows, so the column mean is a warp-shuffle
//                    reduction and the only shared-memory traffic is tile in (16 KB) + hi/lo out (32 KB).
//   MMA thread    : H += hi.hi^T, X += hi.lo^T   (3xTF32 with the third product lo.hi^T = X^T recovered by
//                    symmetry: the partial tile carries 2X and cost_finalize_kernel averages it with its
//                    transpose; 8 instead of 12 MMAs per k-block; fp32 accumulate in TMEM).  The tensor
//                    core's fp32 accumulation truncates, so a long chain into one large accumulator
//                    (e.g. D_ii ~ |x_i|^2 for a fake that resembles its real) picks up a bias that grows
//                    with chain length x magnitude.  The hi.hi products are therefore dealt round-robin
//                    to three TMEM accumulators and the (2^-11 smaller) cross products go to a fourth;
//                    the epilogue adds the four in fp32 (measured: 9x smaller error on video-like data).
//   Timeline (clock64 instrumentation of one CTA, config 2): ~3 us before the first TMA issue (launch, barrier
//                    and TMEM setup), 2 us until the first box lands, 26 boxes x ~1 100 cycles, 3.7 us epilogue.
//                    The per-box time is shared-memory bandwidth: 16 KB TMA in + 16 KB converter reads + 32 KB
//                    hi / lo out + 64 KB of MMA operand reads = 128 KB through a 128 B/clk port.  Splitting the
//                    converter into 2 or 4 groups working on different boxes (8 or 16 warps) did not change it.
//   epilogue      : P'_ij = n_i + n_j - 2 (H_ij + 2 X_ij)  ->  part[p][ks][128][128]  (partial squared
//                    distances up to the symmetrisation; cost_finalize_kernel sums the slabs in fp64,
//                    forms (P'_ij + P'_ji) / 2 and adds the martingale terms).
#include "cost.cuh"
#include "tc_common.cuh"

namespace kccot {

namespace {
constexpr int kRows = 128;
constexpr int kKB = 32;                         // fp32 columns per k-block (one 128-B swizzle row)
constexpr int kTileBytes = kRows * kKB * 4;     // 16 KB
constexpr int kStages = 6;
// bf16 videos: a [R x 32] bf16 box (8 KB, 64-byte swizzle) lands in a staging ring of its own and the converters
// widen it into S.hi / S.lo; 6 stages plus that ring would not fit, 5 do (~206 KB)
constexpr int kStagesBf16 = 5;
constexpr int kStgBytes = kRows * kKB * 2;      // 8 KB
constexpr int kConvWarps = 8;
constexpr int kConvThreads = kConvWarps * 32;
constexpr int kThreads = 64 + kConvThreads;     // warp 0 TMA, warp 1 MMA, warps 2.. convert/epilogue
constexpr int kTmemCols = 512;                 // 4 accumulators of up to 128 columns
constexpr int kNumAcc = 4;

template <int NS>
struct __align__(1024) SmemT {
  uint8_t hi[NS][kTileBytes];
  uint8_t lo[NS][kTileBytes];
  float nrm_part[kConvWarps][kRows];
  float nrm[kRows];
  uint64_t full[NS], conv[NS], empty[NS];
  uint64_t acc_full, acc_empty;
  uint32_t tmem_base;
};
using Smem = SmemT<kStages>;
using SmemBf16 = SmemT<kStagesBf16>;      // followed by the bf16 staging ring stg[kStagesBf16][kStgBytes]

__device__ __forceinline__ uint2 lds64(uint32_t saddr) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(saddr));
  return v;
}
}  // namespace

__global__ void __launch_bounds__(kThreads, 1)
sqdist_tc_kernel(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ CUtensorMap tmy, int Bx, int By,
                 long long K, int nprob, int ksplit, int kbps, float* __restrict__ part, int ctx_period, int ctx_len) {
  extern __shared__ uint8_t smem_raw[];
  // align by OFFSET (not by integer round-trip of the pointer) so that the compiler keeps the shared
  // address space and emits LDS/STS instead of generic LD/ST
  Smem& S = *reinterpret_cast<Smem*>(smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int R = Bx + By;
  const int N = (R + 15) & ~15;
  const int nkb = (int)((K + kKB - 1) / kKB);
  const int nwork = nprob * ksplit;

  if (threadIdx.x == 0) {
    tc::prefetch_tmap(&tmx);
    if (By) tc::prefetch_tmap(&tmy);
    for (int s = 0; s < kStages; ++s) {
      tc::mbar_init(&S.full[s], 1);
      tc::mbar_init(&S.conv[s], kConvWarps);
      tc::mbar_init(&S.empty[s], 1);
    }
    tc::mbar_init(&S.acc_full, 1);
    tc::mbar_init(&S.acc_empty, kConvWarps);
    tc::fence_barrier_init();
  }
  if (warp == 1) {
    tc::tmem_alloc(&S.tmem_base, kTmemCols);
    tc::tmem_relinquish();
  }
  // rows >= R of every stage are never written again: zero them once so the MMA reads zeros
  if (R < kRows)                                           // (nothing to clear when all 128 rows are loaded)
    for (int i = threadIdx.x; i < 2 * kStages * kTileBytes / 16; i += kThreads)
      reinterpret_cast<uint4*>(&S.hi[0][0])[i] = make_uint4(0, 0, 0, 0);
  tc::fence_proxy_async_smem();
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = S.tmem_base;
  pdl_launch_dependents();       // launched with a full dependency: lets cost_finalize_kernel's CTAs take their seats

  if (warp == 0) {
    // ------------------------------- TMA producer ---------------------------------------------
    if (tc::elect_one()) {
      int stage = 0, phase = 0;
      for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
        const int p = w / ksplit, ks = w % ksplit;
        const int kb0 = ks * kbps, kb1 = min(nkb, kb0 + kbps);
        for (int kb = kb0; kb < kb1; ++kb) {
          tc::mbar_wait(&S.empty[stage], phase ^ 1);
          tc::mbar_arrive_expect_tx(&S.full[stage], (uint32_t)R * kKB * 4);
          tc::tma_load_3d(&tmx, &S.full[stage], &S.hi[stage][0], kb * kKB, 0, p);
          // shared-context k-blocks: the fake rows equal the real rows, which were requested one instruction ago
          // (an L2 hit): the fake video's context columns are never read from HBM
          const bool shared = ctx_len != 0 && (kb % ctx_period) < ctx_len;
          if (By) tc::tma_load_3d(shared ? &tmx : &tmy, &S.full[stage], &S.hi[stage][Bx * kKB * 4], kb * kKB, 0, p);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
      // drain the asynchronous tcgen05.commit arrivals on empty[] before the CTA may exit (see grad_tcgen05.cu)
      for (int i = 0; i < kStages; ++i) {
        tc::mbar_wait(&S.empty[stage], phase ^ 1);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------- MMA issuer -----------------------------------------------
    if (tc::elect_one()) {
      const uint32_t idesc = tc::make_idesc_tf32(128, N, 0, 0);
      int stage = 0, phase = 0, acc_phase = 0;
      for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
        const int ks = w % ksplit;
        const int kb0 = ks * kbps, kb1 = min(nkb, kb0 + kbps);
        tc::mbar_wait(&S.acc_empty, acc_phase ^ 1);
        tc::tc_fence_after();
        for (int kb = kb0; kb < kb1; ++kb) {
          tc::mbar_wait(&S.conv[stage], phase);
          tc::tc_fence_after();
          const uint32_t hi_addr = tc::smem_u32(&S.hi[stage][0]);
          const uint32_t lo_addr = tc::smem_u32(&S.lo[stage][0]);
#pragma unroll
          for (int k4 = 0; k4 < kKB / 8; ++k4) {
            const uint64_t dh = tc::make_smem_desc_sw128(hi_addr + k4 * 32, 16, 1024);
            const uint64_t dl = tc::make_smem_desc_sw128(lo_addr + k4 * 32, 16, 1024);
            const int step = (kb - kb0) * (kKB / 8) + k4;
            tc::umma_tf32(tmem + (uint32_t)((step % 3) * kRows), dh, dh, idesc, step >= 3 ? 1u : 0u);
            tc::umma_tf32(tmem + (uint32_t)(3 * kRows), dh, dl, idesc, step > 0 ? 1u : 0u);
          }
          tc::umma_commit(&S.empty[stage]);
          if (kb == kb1 - 1) tc::umma_commit(&S.acc_full);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        acc_phase ^= 1;
      }
    }
  } else {
    // ------------------------------- convert + epilogue ---------------------------------------
    // Converter warp cw owns the 16-byte chunk (4 columns) cw of every row; lane l handles rows
    // l, l+32, l+64, l+96.  A quarter-warp touches 8 consecutive rows, whose swizzled chunk positions
    // are all different: conflict-free.  Column sums are a pure warp reduction (no smem, no barrier).
    const int ct = threadIdx.x - 64;
    const int cw = ct >> 5;
    const int chunk = cw;
    const float invR = 1.f / (float)R;
    int stage = 0, phase = 0, acc_phase = 0;
    for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
      const int ks = w % ksplit;
      const int kb0 = ks * kbps, kb1 = min(nkb, kb0 + kbps);
      float nacc[4] = {0.f, 0.f, 0.f, 0.f};
      for (int kb = kb0; kb < kb1; ++kb) {
        tc::mbar_wait(&S.full[stage], phase);
        const uint32_t hi = tc::smem_u32(&S.hi[stage][0]);
        const uint32_t lo = tc::smem_u32(&S.lo[stage][0]);
        float4 v[4];
        float4 cs = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          const int r = lane + 32 * m;
          v[m] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (r < R) v[m] = tc::lds128(hi + r * 128 + ((chunk ^ (r & 7)) << 4));
          cs.x += v[m].x; cs.y += v[m].y; cs.z += v[m].z; cs.w += v[m].w;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          cs.x += __shfl_xor_sync(0xffffffffu, cs.x, o);
          cs.y += __shfl_xor_sync(0xffffffffu, cs.y, o);
          cs.z += __shfl_xor_sync(0xffffffffu, cs.z, o);
          cs.w += __shfl_xor_sync(0xffffffffu, cs.w, o);
        }
        const long long col0 = (long long)kb * kKB + chunk * 4;
        float4 cen;     // column mean; 0 beyond K so that TMA's zero fill stays zero
        cen.x = (col0 + 0 < K) ? cs.x * invR : 0.f;
        cen.y = (col0 + 1 < K) ? cs.y * invR : 0.f;
        cen.z = (col0 + 2 < K) ? cs.z * invR : 0.f;
        cen.w = (col0 + 3 < K) ? cs.w * invR : 0.f;
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          const int r = lane + 32 * m;
          if (r < R) {
            const float a0 = v[m].x - cen.x, a1 = v[m].y - cen.y, a2 = v[m].z - cen.z, a3 = v[m].w - cen.w;
            nacc[m] = fmaf(a0, a0, fmaf(a1, a1, fmaf(a2, a2, fmaf(a3, a3, nacc[m]))));
            float4 h, l;
            h.x = tc::to_tf32(a0); h.y = tc::to_tf32(a1); h.z = tc::to_tf32(a2); h.w = tc::to_tf32(a3);
            l.x = tc::to_tf32(a0 - h.x); l.y = tc::to_tf32(a1 - h.y);
            l.z = tc::to_tf32(a2 - h.z); l.w = tc::to_tf32(a3 - h.w);
            const int off = r * 128 + ((chunk ^ (r & 7)) << 4);
            tc::sts128(hi + off, h);
            tc::sts128(lo + off, l);
          }
        }
        tc::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&S.conv[stage]);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      // ---- epilogue: row norms -> smem, accumulator -> registers -> partial distances ----------
#pragma unroll
      for (int m = 0; m < 4; ++m) S.nrm_part[cw][lane + 32 * m] = nacc[m];
      tc::named_bar_sync(1, kConvThreads);
      if (ct < kRows) {
        float a = 0.f;
#pragma unroll
        for (int q = 0; q < kConvWarps; ++q) a += S.nrm_part[q][ct];      // fixed order: deterministic
        S.nrm[ct] = a;
      }
      tc::named_bar_sync(1, kConvThreads);
      tc::mbar_wait(&S.acc_full, acc_phase);
      tc::tc_fence_after();
      const int quad = warp & 3;                  // TMEM lane quadrant this warp may read
      const int row = quad * 32 + lane;
      const int half = cw >> 2;                   // columns [64*half, 64*half + 64)
      const float nr = (row < R) ? S.nrm[row] : 0.f;
      // tile-major layout: the ksplit partials of one 8 x 8 output tile are contiguous (ksplit x 256 bytes),
      // so cost_finalize_tiled_kernel reads them as one coalesced stream
      const int pw = w / ksplit;
      float* out = part + ((long long)pw * 256 + (row >> 3) * 16) * ksplit * 64 + (long long)ks * 64 + (row & 7) * 8;
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const int c0 = half * 64 + cc * 32;
        if (c0 < N) {
          float d[32];
          tc::tmem_ld_32x32(tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0, d);
          tc::tmem_ld_wait();
          const int nacc_used = min(kNumAcc - 1, (kb1 - kb0) * (kKB / 8));
          for (int a = 1; a < kNumAcc; ++a) {
            if (a < kNumAcc - 1 && a >= nacc_used) continue;      // accumulator never written in this item
            float t[32];
            tc::tmem_ld_32x32(tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(a * kRows + c0), t);
            tc::tmem_ld_wait();
            const float wt = (a == kNumAcc - 1) ? 2.f : 1.f;          // X stands for X + X^T (see finalize)
#pragma unroll
            for (int j = 0; j < 32; ++j) d[j] = fmaf(wt, t[j], d[j]);
          }
          if (row < R) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              float4 o;
              o.x = nr + S.nrm[min(c0 + j + 0, kRows - 1)] - 2.f * d[j + 0];
              o.y = nr + S.nrm[min(c0 + j + 1, kRows - 1)] - 2.f * d[j + 1];
              o.z = nr + S.nrm[min(c0 + j + 2, kRows - 1)] - 2.f * d[j + 2];
              o.w = nr + S.nrm[min(c0 + j + 3, kRows - 1)] - 2.f * d[j + 3];
              if (c0 + j < R)
                *reinterpret_cast<float4*>(out + (long long)((c0 + j) >> 3) * ksplit * 64 + ((c0 + j) & 7)) = o;
            }
          }
        }
      }
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&S.acc_empty);
      acc_phase ^= 1;
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 1) tc::tmem_dealloc(tmem, kTmemCols);
}

// bf16 videos (raw bits): sqdist_tc_kernel with another load side.  The [R x 32] bf16 box (8 KB, 64-byte swizzle)
// lands in a staging ring of its own and the converters widen it on read (exact); from there on every instruction
// is that of sqdist_tc_kernel, so the partials are bit-identical to the fp32 kernel's on the widened videos.  A
// separate kernel rather than a shared template body: the fp32 kernel keeps its instructions as measured.
__global__ void __launch_bounds__(kThreads, 1)
sqdist_tc_bf16_kernel(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ CUtensorMap tmy, int Bx, int By,
                      long long K, int nprob, int ksplit, int kbps, float* __restrict__ part, int ctx_period,
                      int ctx_len) {
  constexpr int kStages = kStagesBf16;
  extern __shared__ uint8_t smem_raw[];
  SmemBf16& S = *reinterpret_cast<SmemBf16*>(smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u));
  uint8_t* stg = reinterpret_cast<uint8_t*>(&S) + sizeof(SmemBf16);     // staging ring [kStages][kStgBytes]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int R = Bx + By;
  const int N = (R + 15) & ~15;
  const int nkb = (int)((K + kKB - 1) / kKB);
  const int nwork = nprob * ksplit;

  if (threadIdx.x == 0) {
    tc::prefetch_tmap(&tmx);
    if (By) tc::prefetch_tmap(&tmy);
    for (int s = 0; s < kStages; ++s) {
      tc::mbar_init(&S.full[s], 1);
      tc::mbar_init(&S.conv[s], kConvWarps);
      tc::mbar_init(&S.empty[s], 1);
    }
    tc::mbar_init(&S.acc_full, 1);
    tc::mbar_init(&S.acc_empty, kConvWarps);
    tc::fence_barrier_init();
  }
  if (warp == 1) {
    tc::tmem_alloc(&S.tmem_base, kTmemCols);
    tc::tmem_relinquish();
  }
  // rows >= R of every stage are never written again: zero them once so the MMA reads zeros
  if (R < kRows)                                           // (nothing to clear when all 128 rows are loaded)
    for (int i = threadIdx.x; i < 2 * kStages * kTileBytes / 16; i += kThreads)
      reinterpret_cast<uint4*>(&S.hi[0][0])[i] = make_uint4(0, 0, 0, 0);
  tc::fence_proxy_async_smem();
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = S.tmem_base;
  pdl_launch_dependents();       // launched with a full dependency: lets cost_finalize_kernel's CTAs take their seats

  if (warp == 0) {
    // ------------------------------- TMA producer ---------------------------------------------
    if (tc::elect_one()) {
      int stage = 0, phase = 0;
      for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
        const int p = w / ksplit, ks = w % ksplit;
        const int kb0 = ks * kbps, kb1 = min(nkb, kb0 + kbps);
        for (int kb = kb0; kb < kb1; ++kb) {
          tc::mbar_wait(&S.empty[stage], phase ^ 1);
          uint8_t* dst = stg + (size_t)stage * kStgBytes;
          tc::mbar_arrive_expect_tx(&S.full[stage], (uint32_t)R * kKB * 2);
          tc::tma_load_3d(&tmx, &S.full[stage], dst, kb * kKB, 0, p);
          const bool shared = ctx_len != 0 && (kb % ctx_period) < ctx_len;      // shared-context k-blocks
          if (By) tc::tma_load_3d(shared ? &tmx : &tmy, &S.full[stage], dst + Bx * kKB * 2, kb * kKB, 0, p);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
      // drain the asynchronous tcgen05.commit arrivals on empty[] before the CTA may exit (see grad_tcgen05.cu)
      for (int i = 0; i < kStages; ++i) {
        tc::mbar_wait(&S.empty[stage], phase ^ 1);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------- MMA issuer -----------------------------------------------
    if (tc::elect_one()) {
      const uint32_t idesc = tc::make_idesc_tf32(128, N, 0, 0);
      int stage = 0, phase = 0, acc_phase = 0;
      for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
        const int ks = w % ksplit;
        const int kb0 = ks * kbps, kb1 = min(nkb, kb0 + kbps);
        tc::mbar_wait(&S.acc_empty, acc_phase ^ 1);
        tc::tc_fence_after();
        for (int kb = kb0; kb < kb1; ++kb) {
          tc::mbar_wait(&S.conv[stage], phase);
          tc::tc_fence_after();
          const uint32_t hi_addr = tc::smem_u32(&S.hi[stage][0]);
          const uint32_t lo_addr = tc::smem_u32(&S.lo[stage][0]);
#pragma unroll
          for (int k4 = 0; k4 < kKB / 8; ++k4) {
            const uint64_t dh = tc::make_smem_desc_sw128(hi_addr + k4 * 32, 16, 1024);
            const uint64_t dl = tc::make_smem_desc_sw128(lo_addr + k4 * 32, 16, 1024);
            const int step = (kb - kb0) * (kKB / 8) + k4;
            tc::umma_tf32(tmem + (uint32_t)((step % 3) * kRows), dh, dh, idesc, step >= 3 ? 1u : 0u);
            tc::umma_tf32(tmem + (uint32_t)(3 * kRows), dh, dl, idesc, step > 0 ? 1u : 0u);
          }
          tc::umma_commit(&S.empty[stage]);
          if (kb == kb1 - 1) tc::umma_commit(&S.acc_full);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        acc_phase ^= 1;
      }
    }
  } else {
    // ------------------------------- convert + epilogue ---------------------------------------
    // Converter warp cw owns the 16-byte chunk (4 columns) cw of every row; lane l handles rows
    // l, l+32, l+64, l+96.  A quarter-warp touches 8 consecutive rows, whose swizzled chunk positions
    // are all different: conflict-free.  Column sums are a pure warp reduction (no smem, no barrier).
    const int ct = threadIdx.x - 64;
    const int cw = ct >> 5;
    const int chunk = cw;
    const float invR = 1.f / (float)R;
    int stage = 0, phase = 0, acc_phase = 0;
    for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
      const int ks = w % ksplit;
      const int kb0 = ks * kbps, kb1 = min(nkb, kb0 + kbps);
      float nacc[4] = {0.f, 0.f, 0.f, 0.f};
      for (int kb = kb0; kb < kb1; ++kb) {
        tc::mbar_wait(&S.full[stage], phase);
        const uint32_t hi = tc::smem_u32(&S.hi[stage][0]);
        const uint32_t lo = tc::smem_u32(&S.lo[stage][0]);
        const uint32_t sb = tc::smem_u32(stg + (size_t)stage * kStgBytes);
        float4 v[4];
        float4 cs = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          const int r = lane + 32 * m;
          v[m] = make_float4(0.f, 0.f, 0.f, 0.f);
          // 64-byte swizzle: 16-byte unit (chunk / 2) of row r sits at position (chunk / 2) ^ ((r / 2) % 4)
          if (r < R) v[m] = widen_bf16x4(lds64(sb + r * 64 + ((((chunk >> 1) ^ ((r >> 1) & 3)) << 4) | ((chunk & 1) << 3))));
          cs.x += v[m].x; cs.y += v[m].y; cs.z += v[m].z; cs.w += v[m].w;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          cs.x += __shfl_xor_sync(0xffffffffu, cs.x, o);
          cs.y += __shfl_xor_sync(0xffffffffu, cs.y, o);
          cs.z += __shfl_xor_sync(0xffffffffu, cs.z, o);
          cs.w += __shfl_xor_sync(0xffffffffu, cs.w, o);
        }
        const long long col0 = (long long)kb * kKB + chunk * 4;
        float4 cen;     // column mean; 0 beyond K so that TMA's zero fill stays zero
        cen.x = (col0 + 0 < K) ? cs.x * invR : 0.f;
        cen.y = (col0 + 1 < K) ? cs.y * invR : 0.f;
        cen.z = (col0 + 2 < K) ? cs.z * invR : 0.f;
        cen.w = (col0 + 3 < K) ? cs.w * invR : 0.f;
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          const int r = lane + 32 * m;
          if (r < R) {
            const float a0 = v[m].x - cen.x, a1 = v[m].y - cen.y, a2 = v[m].z - cen.z, a3 = v[m].w - cen.w;
            nacc[m] = fmaf(a0, a0, fmaf(a1, a1, fmaf(a2, a2, fmaf(a3, a3, nacc[m]))));
            float4 h, l;
            h.x = tc::to_tf32(a0); h.y = tc::to_tf32(a1); h.z = tc::to_tf32(a2); h.w = tc::to_tf32(a3);
            l.x = tc::to_tf32(a0 - h.x); l.y = tc::to_tf32(a1 - h.y);
            l.z = tc::to_tf32(a2 - h.z); l.w = tc::to_tf32(a3 - h.w);
            const int off = r * 128 + ((chunk ^ (r & 7)) << 4);
            tc::sts128(hi + off, h);
            tc::sts128(lo + off, l);
          }
        }
        tc::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&S.conv[stage]);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      // ---- epilogue: row norms -> smem, accumulator -> registers -> partial distances ----------
#pragma unroll
      for (int m = 0; m < 4; ++m) S.nrm_part[cw][lane + 32 * m] = nacc[m];
      tc::named_bar_sync(1, kConvThreads);
      if (ct < kRows) {
        float a = 0.f;
#pragma unroll
        for (int q = 0; q < kConvWarps; ++q) a += S.nrm_part[q][ct];      // fixed order: deterministic
        S.nrm[ct] = a;
      }
      tc::named_bar_sync(1, kConvThreads);
      tc::mbar_wait(&S.acc_full, acc_phase);
      tc::tc_fence_after();
      const int quad = warp & 3;                  // TMEM lane quadrant this warp may read
      const int row = quad * 32 + lane;
      const int half = cw >> 2;                   // columns [64*half, 64*half + 64)
      const float nr = (row < R) ? S.nrm[row] : 0.f;
      // tile-major layout: the ksplit partials of one 8 x 8 output tile are contiguous (ksplit x 256 bytes),
      // so cost_finalize_tiled_kernel reads them as one coalesced stream
      const int pw = w / ksplit;
      float* out = part + ((long long)pw * 256 + (row >> 3) * 16) * ksplit * 64 + (long long)ks * 64 + (row & 7) * 8;
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const int c0 = half * 64 + cc * 32;
        if (c0 < N) {
          float d[32];
          tc::tmem_ld_32x32(tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0, d);
          tc::tmem_ld_wait();
          const int nacc_used = min(kNumAcc - 1, (kb1 - kb0) * (kKB / 8));
          for (int a = 1; a < kNumAcc; ++a) {
            if (a < kNumAcc - 1 && a >= nacc_used) continue;      // accumulator never written in this item
            float t[32];
            tc::tmem_ld_32x32(tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(a * kRows + c0), t);
            tc::tmem_ld_wait();
            const float wt = (a == kNumAcc - 1) ? 2.f : 1.f;          // X stands for X + X^T (see finalize)
#pragma unroll
            for (int j = 0; j < 32; ++j) d[j] = fmaf(wt, t[j], d[j]);
          }
          if (row < R) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              float4 o;
              o.x = nr + S.nrm[min(c0 + j + 0, kRows - 1)] - 2.f * d[j + 0];
              o.y = nr + S.nrm[min(c0 + j + 1, kRows - 1)] - 2.f * d[j + 1];
              o.z = nr + S.nrm[min(c0 + j + 2, kRows - 1)] - 2.f * d[j + 2];
              o.w = nr + S.nrm[min(c0 + j + 3, kRows - 1)] - 2.f * d[j + 3];
              if (c0 + j < R)
                *reinterpret_cast<float4*>(out + (long long)((c0 + j) >> 3) * ksplit * 64 + ((c0 + j) & 7)) = o;
            }
          }
        }
      }
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&S.acc_empty);
      acc_phase ^= 1;
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 1) tc::tmem_dealloc(tmem, kTmemCols);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

int encode_tmap_3d(CUtensorMap* out, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes,
                   uint64_t stride2_bytes, uint32_t b0, uint32_t b1, bool atom32, bool noswizzle) {
  return encode_tmap_3d(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32,
                        noswizzle ? CU_TENSOR_MAP_SWIZZLE_NONE
                                  : (atom32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B),
                        base, d0, d1, d2, stride1_bytes, stride2_bytes, b0, b1);
}

int encode_tmap_3d(CUtensorMap* out, CUtensorMapDataType dtype, CUtensorMapSwizzle swizzle, const void* base,
                   uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t b0,
                   uint32_t b1) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled entry point not available");
    return KCCOT_ECUDA;
  }
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
  cuuint32_t box[3] = {b0, b1, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(out, dtype, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (dims %llu x %llu x %llu, box %u x %u)", (int)r,
              (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2, b0, b1);
    return KCCOT_ECUDA;
  }
  return KCCOT_OK;
}

int encode_tmap_2d_f16(CUtensorMap* out, const void* base, uint64_t cols, uint64_t rows, uint64_t pitch_bytes,
                       uint32_t box_cols, uint32_t box_rows) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled entry point not available");
    return KCCOT_ECUDA;
  }
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {pitch_bytes};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (fp16 2-D) failed with CUresult %d (dims %llu x %llu, pitch %llu, box %u x %u)", (int)r,
              (unsigned long long)cols, (unsigned long long)rows, (unsigned long long)pitch_bytes, box_cols, box_rows);
    return KCCOT_ECUDA;
  }
  return KCCOT_OK;
}

bool tc_sqdist_supported(const float* x, const float* y, int Bx, int By, long long K) {
  const int R = Bx + (y ? By : 0);
  if (R > kRows || Bx % 8 != 0 || (y && By % 8 != 0)) return false;
  if (K % 4 != 0 || K < kKB) return false;
  if ((reinterpret_cast<uintptr_t>(x) & 15) || (y && (reinterpret_cast<uintptr_t>(y) & 15))) return false;
  return true;
}

void tc_sqdist_plan(int nprob, int R, long long K, int* ksplit, int* kbps) {
  (void)R;
  const int nkb = (int)((K + kKB - 1) / kKB);
  const int sms = num_sms();
  // pick the split whose work-item count wastes the fewest CTA slots in the last wave, keeping
  // at least 8 k-blocks (128 KB of input) per item so the 64 KB partial tile stays amortised
  int best = 1;
  double best_eff = 0.0;
  const int max_split = max(1, min(nkb / 8, (8 * sms + nprob - 1) / nprob));
  for (int s = 1; s <= max_split; ++s) {
    const long long work = (long long)nprob * s;
    const long long waves = (work + sms - 1) / sms;
    const double eff = (double)work / (double)(waves * sms);
    if (eff > best_eff + 1e-9) { best_eff = eff; best = s; }
    if (work >= sms && eff > 0.97) break;
  }
  int per = (nkb + best - 1) / best;
  *ksplit = (nkb + per - 1) / per;
  *kbps = per;
}

int launch_sqdist_partials_tc(const float* x, const float* y, int nprob, int Bx, int By, long long K, int ksplit,
                              int kbps, float* part, cudaStream_t st) {
  CUtensorMap tmx, tmy;
  int rc = encode_tmap_3d(&tmx, x, (uint64_t)K, (uint64_t)Bx, (uint64_t)nprob, (uint64_t)K * 4,
                          (uint64_t)K * 4 * Bx, kKB, (uint32_t)Bx);
  if (rc) return rc;
  if (y) {
    rc = encode_tmap_3d(&tmy, y, (uint64_t)K, (uint64_t)By, (uint64_t)nprob, (uint64_t)K * 4, (uint64_t)K * 4 * By,
                        kKB, (uint32_t)By);
    if (rc) return rc;
  } else {
    tmy = tmx;
    By = 0;
  }
  const size_t smem = sizeof(Smem) + 1024;
  static size_t attr_set[kMaxDevices] = {};
  if (smem_attr_needed(attr_set, smem))
    KCCOT_CUDA(cudaFuncSetAttribute(sqdist_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int grid = min(nprob * ksplit, num_sms());
  int ctx_period = 0, ctx_len = 0;
  if (!(By && Bx == By && ctx_boxes(K, &ctx_period, &ctx_len))) ctx_period = ctx_len = 0;
  sqdist_tc_kernel<<<grid, kThreads, smem, st>>>(tmx, tmy, Bx, By, K, nprob, ksplit, kbps, part, ctx_period, ctx_len);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}

bool tc_sqdist_bf16_supported(int Bx, int By, long long K) {
  return Bx + By <= kRows && Bx % 8 == 0 && By % 8 == 0 && K % 8 == 0 && K >= kKB;
}

// bf16 videos (raw bits, 16-byte aligned rows, K % 8 == 0): [R x 32] bf16 boxes with the 64-byte swizzle the
// converters read; same plan, same partials as launch_sqdist_partials_tc on the widened copies
int launch_sqdist_partials_tc_bf16(const uint16_t* x, const uint16_t* y, int nprob, int Bx, int By, long long K,
                                   int ksplit, int kbps, float* part, cudaStream_t st) {
  CUtensorMap tmx, tmy;
  if (int rc = encode_tmap_3d(&tmx, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, CU_TENSOR_MAP_SWIZZLE_64B, x, (uint64_t)K,
                              (uint64_t)Bx, (uint64_t)nprob, (uint64_t)K * 2, (uint64_t)K * 2 * Bx, kKB, (uint32_t)Bx))
    return rc;
  if (int rc = encode_tmap_3d(&tmy, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, CU_TENSOR_MAP_SWIZZLE_64B, y, (uint64_t)K,
                              (uint64_t)By, (uint64_t)nprob, (uint64_t)K * 2, (uint64_t)K * 2 * By, kKB, (uint32_t)By))
    return rc;
  const size_t smem = sizeof(SmemBf16) + (size_t)kStagesBf16 * kStgBytes + 1024;
  static size_t attr_set[kMaxDevices] = {};
  if (smem_attr_needed(attr_set, smem))
    KCCOT_CUDA(cudaFuncSetAttribute(sqdist_tc_bf16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int grid = min(nprob * ksplit, num_sms());
  int ctx_period = 0, ctx_len = 0;
  if (!(Bx == By && ctx_boxes(K, &ctx_period, &ctx_len))) ctx_period = ctx_len = 0;
  sqdist_tc_bf16_kernel<<<grid, kThreads, smem, st>>>(tmx, tmy, Bx, By, K, nprob, ksplit, kbps, part, ctx_period,
                                                       ctx_len);
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}

}  // namespace kccot
