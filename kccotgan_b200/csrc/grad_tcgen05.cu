// Adjoint of the squared-distance cost on the tensor cores.
//
// With the stacked rows z = [x; y] (R = Bx + By <= 128) and a weight matrix W [R,R] built from the
// adjoints of the cost matrices, every wanted gradient row is
//     g_r = 2s * sum_c W_rc (z_r - z_c) = -2s * sum_c W'_rc z_c,   W' = W - diag(rowsum(W)),
// i.e. a skinny GEMM  G[r, col] = sum_c W'[r, c] * Z[c, col]  streamed once over the video columns.
//
//   A operand = W', split tf32 hi/lo ONCE per launch by build_w_image_kernel (a 64-block kernel in front) and parked
//               in TENSOR MEMORY by every CTA (TS-mode tcgen05.mma: lane = A row, column = contraction index).  An
//               SS-mode M=128 x N=64 x K=8 instruction re-reads 4 KB of A + 2 KB of B from shared memory per 32
//               cycles of math (~190 B/clk against a 128 B/clk port, measured as the wall with the clock64
//               timeline); with A in TMEM only B touches shared memory.
//               The launch produces at most 64 output rows, so the 128 A rows of the M = 128 instruction hold BOTH
//               halves of the split: in every 32-lane quadrant q, lanes 0-15 carry W'hi of output rows 16q..16q+15 and
//               lanes 16-31 carry W'lo of the same rows.  One instruction then yields W'hi.[Zhi | Zlo] and W'lo.Zhi
//               at once (the fourth block, W'lo.Zlo, is 2^-22 of the result and is dropped by the epilogue).
//   B operand = the TMA-loaded video box itself, N-major ("MN-major"): a [rows x 32] fp32 box.  tcgen05
//               accepts exactly one shared-memory layout for MN-major 32-bit operands,
//               SWIZZLE_128B_BASE32B (32-byte chunks XOR row%4, 4-row atoms, SBO = 512 B); the boxes
//               are loaded with the matching TMA mode 128B_ATOM_32B, so no transposition is needed.
//               B = [Zhi | Zlo]: two N-atoms, LBO = distance between the hi and lo rings.  kind::tf32 reads fp32
//               words and IGNORES the low 13 mantissa bits, so the raw box serves as Zhi = trunc(Z) as it stands; the
//               converter warps only write Zlo = Z - trunc(Z) (exact in fp32) into the lo ring.
//   Stage     = ONE box (8 KB + 8 KB lo at 64 rows): the ring is 5 deep, and with two CTAs per SM 10 boxes are in
//               flight per SM, which is what hides the HBM latency (the first version used two 64 KB stages and
//               starved 44 % of the time).
//   3xTF32 in ONE instruction per k-step (M = 128, N = 64, K = 8).  The elected lane needs ~30-40 cycles per
//               tcgen05.mma (descriptor moves to uniform registers; measured with the clock64 timeline) and the
//               earlier two-instruction form (N = 64 for W'hi, N = 32 for W'lo, converter rewriting the hi box
//               rounded) was shared-memory bound: 136 KB through the port per 24 KB tile (TMA write, converter read /
//               write, operand reads, output staging), 1 420 cycles per tile.  This one moves 96 KB and its steady
//               state is the HBM itself: ~1 100 cycles per tile = 22 B/clk per SM = the measured copy peak.  fp32
//               accumulate in TMEM, 2 accumulator buffers of 64 columns (256 columns with W': half of an SM's).
//   Epilogue:   each of the four epilogue warps owns one quadrant: lanes 0-15 add their two column halves, lanes
//               16-31 hand W'lo.Zhi down by shuffle; 16 rows per warp are staged in 128-byte-swizzled shared memory
//               and one TMA store (or reduce-add) writes the [N x 32] box as full 128-byte row segments.
#include "cost.cuh"
#include "tc_common.cuh"

namespace kccot {

namespace {
constexpr int kCols = 32;                  // video columns per work tile (UMMA N) = one TMA box
constexpr int kBoxCols = 32;               // fp32 columns per TMA box (128-byte swizzle row)
constexpr int kMaxN = 64;                  // output rows per launch
// Half-SM footprint: two CTAs fit on one SM (shared memory, registers and tensor memory), so a CTA of another
// evaluation streams while this one sets up or drains.  Two CTAs keep 2 x 5 boxes in flight per SM.
constexpr int kStages = 5;
constexpr int kConvWarps = kStages;         // ONE converter warp per ring slot (see the converter branch for why)
constexpr int kConvThreads = kConvWarps * 32;
constexpr int kEpiWarps = 4;
constexpr int kThreads = 64 + kConvThreads + kEpiWarps * 32;   // 352
constexpr int kCtasPerSm = 2;
constexpr int kAccBufs = 2;                // the epilogue needs ~1 000 of a tile's ~1 100 cycles: two buffers keep up
constexpr int kAccCols = 64;               // per tile: [W.Zhi | W.Zlo], 32 columns each
constexpr int kTmemCols = 256;             // W' (hi / lo interleaved by lane) [0,128) | 2 accumulator buffers x 64 columns
constexpr int kTmemAcc0 = 128;
constexpr bool kRawHi = true;              // the MMA truncates the raw box itself; converters write only the lo box
constexpr int kObufBytes = kMaxN * 128;     // one staged output tile
static_assert(kTmemCols >= kTmemAcc0 + kAccBufs * kAccCols && kTmemCols * kCtasPerSm <= 512, "tensor memory");

struct Bars {
  uint64_t full[kStages], conv[kStages], empty[kStages];
  uint64_t acc_full[kAccBufs], acc_empty[kAccBufs];
  uint64_t w_ready;                          // W' is in tensor memory (4 loader warps arrive)
  uint32_t tmem_base;
};

// W' image builder.  One block per (output row rr < 64, row block rb, problem): thread c forms W'[r][c] of the stacked
// weight matrix (r = row_off + rr; row block 0 = the x rows, 1 = the y rows), the block reduces the row sum (diagonal
// = -sum), splits into tf32 hi + lo and writes both into the TENSOR-MEMORY IMAGE the gradient kernel loads:
//     img[p][rb][c / 4][lane][c % 4],  lane = 32 (rr / 16) + (rr % 16) for the hi part, + 16 for the lo part
// (lane-contiguous 16-byte units: a warp of the gradient kernel reads 512 contiguous bytes per load).  Rows rr >= N and
// columns c >= R are zero.  148 gradient CTAs used to build the same W' each (~9 600 cycles before their first MMA,
// arithmetic-bound on four warps); now they copy 64 KB from L2.
//   kMixed: C = Cbar3 [nprob,3,B,B] (xy, xx, yy; weights already applied):
//       x-row r:  [ Cxx[r][c] + Cxx[c][r] | Cxy[r][c'] ],   y-row j:  [ Cxy[c][j] | Cyy[j][c'] + Cyy[c'][j] ]
//   else:   C = Cbar [nprob,Bx,By] of one pair:  W'[i][Bx+j] = W'[Bx+j][i] = Cbar_ij
constexpr int kImgFloats = 128 * 128;
template <bool kMixed>
__global__ void __launch_bounds__(128) build_w_image_kernel(const float* __restrict__ C, int Bx, int By, int rb_first,
                                                            float* __restrict__ img) {
  pdl_wait();                    // C comes from the kernel before
  pdl_launch_dependents();       // the gradient kernel's ring fill may start; it waits for this grid before reading img
  const int rr = blockIdx.x, rb = rb_first + blockIdx.y, p = blockIdx.z, c = threadIdx.x;
  const int R = Bx + By;
  const int row_off = rb ? Bx : 0, N = rb ? By : Bx;
  const int r = row_off + rr;
  float w = 0.f;
  if (rr < N && c < R && c != r) {
    if (kMixed) {
      const int B = Bx;
      const long long BB = (long long)B * B;
      const float* Cxy = C + (long long)p * 3 * BB;
      const float* Cxx = Cxy + BB;
      const float* Cyy = Cxy + 2 * BB;
      if (r < B) w = (c < B) ? Cxx[(long long)r * B + c] + Cxx[(long long)c * B + r] : Cxy[(long long)r * B + (c - B)];
      else w = (c < B) ? Cxy[(long long)c * B + (r - B)]
                       : Cyy[(long long)(r - B) * B + (c - B)] + Cyy[(long long)(c - B) * B + (r - B)];
    } else {
      const float* Cp = C + (long long)p * Bx * By;
      if (r < Bx && c >= Bx) w = Cp[(long long)r * By + (c - Bx)];
      else if (r >= Bx && c < Bx) w = Cp[(long long)c * By + (r - Bx)];
    }
  }
  __shared__ float red[4];
  const float s = warp_sum(w);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (c == r && rr < N) w = -(red[0] + red[1] + red[2] + red[3]);
  const float hi = tc::to_tf32(w), lo = tc::to_tf32(w - hi);
  const int lane_hi = 32 * (rr >> 4) + (rr & 15);
  float* im = img + ((long long)p * 2 + rb) * kImgFloats + (long long)(c >> 2) * 512 + (c & 3);
  im[lane_hi * 4] = hi;
  im[(lane_hi + 16) * 4] = lo;
}

// bf16 videos (grad_tc_bf16_kernel): the [rows x 32] bf16 box (rows x 64 B, unswizzled) lands in the LO slot of its
// stage, which is free because a widened bf16 value has Zlo = Z - trunc_tf32(Z) = 0 exactly: the W'hi.Zlo block of
// the fp32 instruction is zero and is not computed.  The slot's converter warp widens the box into the hi slot at the
// SWIZZLE_128B_BASE32B positions the fp32 TMA box would have had, the MMA is M128 x N32 x K8 over Zhi only, and the
// epilogue rounds to bf16 (nearest even) and stores a [N x 32] bf16 box (64-byte swizzle).
__device__ __forceinline__ uint2 lds64(uint32_t saddr) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(saddr));
  return v;
}

template <bool kBf16>
__device__ __forceinline__ void grad_tc_body(const CUtensorMap& tmx, const CUtensorMap& tmy, const CUtensorMap& tmo,
                                             int Bx, int By, long long K, const float* __restrict__ Wimg, int rb, int N,
                                             float neg2s, int accumulate, int ctx_period, int ctx_len) {
  extern __shared__ uint8_t smem_raw[];
  // align by OFFSET so that the compiler keeps the shared address space (LDS/STS, not generic LD/ST)
  uint8_t* base = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rows_max = max(Bx, By);
  const int stage_bytes = rows_max * 128;           // one [rows x 32] box
  // layout: hi[kStages] | lo[kStages] | output staging | barriers   (W' lives in tensor memory)
  uint8_t* st_hi = base;
  uint8_t* st_lo = st_hi + (size_t)kStages * stage_bytes;
  uint8_t* obuf = st_lo + (size_t)kStages * stage_bytes;      // 2 x [64 rows x 128 B] output staging (swizzled)
  Bars& bars = *reinterpret_cast<Bars*>(obuf + 2 * kObufBytes);

  const int p = blockIdx.y;
  // Shared-context hint (ctx_len != 0): the column tiles whose index modulo ctx_period is below ctx_len are skipped
  // altogether (their gradient rows are constants of the caller); the loops run over the ACTIVE tiles and
  // tile_of() maps an active index to its column tile.
  const int ctx_active = ctx_period - ctx_len;
  const long long ntiles_all = (K + kCols - 1) / kCols;
  const long long ntiles = ctx_len ? ntiles_all / ctx_period * ctx_active : ntiles_all;
  auto tile_of = [&](long long i) -> long long {
    return ctx_len ? (i / ctx_active) * ctx_period + ctx_len + (i % ctx_active) : i;
  };
  // each CTA streams a CONTIGUOUS range of column tiles: consecutive 128-byte segments of a row are
  // fetched by the same SM back to back (DRAM page / L2 256-byte promotion locality)
  const long long tpc = (ntiles + gridDim.x - 1) / gridDim.x;
  const long long t_begin = blockIdx.x * tpc, t_end = min(ntiles, t_begin + tpc);

  if (threadIdx.x == 0) {
    tc::prefetch_tmap(&tmx);
    tc::prefetch_tmap(&tmy);
    tc::prefetch_tmap(&tmo);
    for (int s = 0; s < kStages; ++s) {
      tc::mbar_init(&bars.full[s], 1);
      tc::mbar_init(&bars.conv[s], 1);                      // one converter warp per box
      tc::mbar_init(&bars.empty[s], 1);
    }
    for (int b = 0; b < kAccBufs; ++b) {
      tc::mbar_init(&bars.acc_full[b], 1);
      tc::mbar_init(&bars.acc_empty[b], kEpiWarps);         // one arrival per quadrant
    }
    tc::mbar_init(&bars.w_ready, kEpiWarps);
    tc::fence_barrier_init();
  }
  if (warp == 1) {
    tc::tmem_alloc(&bars.tmem_base, kTmemCols);
    tc::tmem_relinquish();
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = bars.tmem_base;
  // W' -> tensor memory, by the four epilogue warps (one 32-lane quadrant each): a straight copy of the image that
  // build_w_image_kernel left in global memory (lane l of quadrant q holds A row 16q + (l & 15): its tf32 hi part on
  // lanes 0-15, its lo part on lanes 16-31).  The TMA producer and the converters do not wait for it: the ring fills
  // meanwhile; only the MMA issuer waits on w_ready.
  if (warp >= 2 + kConvWarps) {
    pdl_wait();      // the image comes from the kernel before; the TMA producer and the converters (videos only) run ahead
    const int quadw = warp & 3;
    const uint32_t ta0 = tmem + ((uint32_t)(quadw * 32) << 16);
    const float4* im = reinterpret_cast<const float4*>(Wimg + ((long long)p * 2 + rb) * kImgFloats) + (quadw * 32 + lane);
#pragma unroll
    for (int h2 = 0; h2 < 2; ++h2) {                        // 64 contraction columns per round: 16 loads in flight
      float a[32], b[32];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 t = im[(h2 * 16 + j) * 128];
        a[4 * j] = t.x; a[4 * j + 1] = t.y; a[4 * j + 2] = t.z; a[4 * j + 3] = t.w;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 t = im[(h2 * 16 + 8 + j) * 128];
        b[4 * j] = t.x; b[4 * j + 1] = t.y; b[4 * j + 2] = t.z; b[4 * j + 3] = t.w;
      }
      tc::tmem_st_32x32(ta0 + (uint32_t)(h2 * 64), a);
      tc::tmem_st_32x32(ta0 + (uint32_t)(h2 * 64 + 32), b);
    }
    tc::tmem_st_wait();
    tc::tc_fence_before();
    __syncwarp();
    if (lane == 0) tc::mbar_arrive(&bars.w_ready);
  }

  if (warp == 0) {
    // ------------------------------- TMA producer ---------------------------------------------
    if (tc::elect_one()) {
      int stage = 0, phase = 0;
      for (long long t = t_begin; t < t_end; ++t) {
        const int col0 = (int)(tile_of(t) * kCols);
        for (int half = 0; half < 2; ++half) {
          const int rows = half ? By : Bx;
          if (rows == 0) continue;
          const CUtensorMap* tm = half ? &tmy : &tmx;
          tc::mbar_wait(&bars.empty[stage], phase ^ 1);
          tc::mbar_arrive_expect_tx(&bars.full[stage], (uint32_t)(rows * (kBf16 ? 64 : 128)));
          tc::tma_load_3d(tm, &bars.full[stage], (kBf16 ? st_lo : st_hi) + (size_t)stage * stage_bytes, col0, 0, p);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
      // Drain: the tcgen05.commit arrivals on empty[] are asynchronous and nobody else waits for the last ones; an
      // arrival must not land after the CTA has exited (the shared memory then belongs to the next CTA on this SM).
      for (int i = 0; i < kStages; ++i) {
        tc::mbar_wait(&bars.empty[stage], phase ^ 1);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------- MMA issuer -----------------------------------------------
    if (tc::elect_one()) {
      const uint32_t idesc = tc::make_idesc_tf32(128, kBf16 ? kCols : kAccCols, /*A K-major*/ 0, /*B MN-major*/ 1);
      const uint32_t lbo = (uint32_t)((size_t)kStages * stage_bytes);     // hi box -> lo box of the same stage
      int stage = 0, phase = 0;
      int ab = 0, ab_phase = 0;
      tc::mbar_wait(&bars.w_ready, 0);
      tc::tc_fence_after();
      for (long long t = t_begin; t < t_end; ++t) {
        tc::mbar_wait(&bars.acc_empty[ab], ab_phase ^ 1);
        tc::tc_fence_after();
        const uint32_t d_tmem = tmem + (uint32_t)(kTmemAcc0 + ab * kAccCols);
        bool first = true;
        for (int half = 0; half < 2; ++half) {
          const int rows = half ? By : Bx;
          if (rows == 0) continue;
          const uint32_t a_w = tmem + (uint32_t)(half ? Bx : 0);           // W' columns of this half
          tc::mbar_wait(&bars.conv[stage], phase);
          tc::tc_fence_after();
          // N-major B over two atoms: columns 0-31 = Zhi box, 32-63 = Zlo box (LBO apart); 4-row swizzle
          // atoms 512 B apart, 8 contraction rows per k-step
          const uint64_t b0 = tc::make_smem_desc(tc::smem_u32(st_hi + (size_t)stage * stage_bytes), lbo, 512, 1);
          const int nk = rows >> 3;
#pragma unroll
          for (int kk = 0; kk < kMaxN / 8; ++kk) {
            if (kk < nk) {
              // lanes 0-15 of each quadrant: [W'hi.Zhi | W'hi.Zlo]; lanes 16-31: [W'lo.Zhi | (W'lo.Zlo)]
              tc::umma_tf32_ts(d_tmem, a_w + kk * 8, b0 + (uint32_t)(kk * 64), idesc, first ? 0u : 1u);
              first = false;
            }
          }
          tc::umma_commit(&bars.empty[stage]);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        tc::umma_commit(&bars.acc_full[ab]);
        if (++ab == kAccBufs) { ab = 0; ab_phase ^= 1; }
      }
    }
  } else if (warp < 2 + kConvWarps) {
    // ------------------------------- tf32 hi / lo split ---------------------------------------
    // Warp-per-SLOT: converter warp cw owns ring slot cw, i.e. the boxes cw, cw + kStages, ... — up to kStages boxes
    // are being converted at once (all warps on one box serialised the boxes at ~600 cycles each).
    // The owner sees EVERY phase of full[cw] in order, which the parity wait needs.  An earlier version dealt the
    // boxes round-robin over 8 warps with 9 slots: after box n a warp went on to box n + 8, which lives in the slot of
    // box n - 1, a box that ANOTHER warp waits for.  TMA loads complete out of order; when box n landed and was
    // converted before box n - 1 had landed, full[slot(n-1)] still showed the phase before box n - 1, whose parity is
    // the one box n + 8 waits for: the wait passed, the warp converted a slot that was being filled and arrived on
    // conv[] a pass early, and the barriers of the ring went out of step for good (the kernel hung about once in a
    // few hundred thousand CTAs; DESIGN.md records how it was found).
    const int cw = warp - 2;
    const int nhalves = (Bx ? 1 : 0) + (By ? 1 : 0);
    const long long nbox = (t_end - t_begin) * nhalves;
    const uint32_t hi = tc::smem_u32(st_hi + (size_t)cw * stage_bytes);
    const uint32_t lo = tc::smem_u32(st_lo + (size_t)cw * stage_bytes);
    int phase = 0;
    for (long long n = cw; n < nbox; n += kStages, phase ^= 1) {
      const int half = nhalves == 2 ? (int)(n & 1) : (Bx ? 0 : 1);
      const int rows = half ? By : Bx;
      tc::mbar_wait(&bars.full[cw], phase);
      const int n16 = rows * 8;                           // 16-byte units in this box (multiple of 64)
      if (kBf16) {
        // unit e = (row r, fp32 chunk j): 8 bytes of bf16 in, 16 bytes of fp32 out at the SWIZZLE_128B_BASE32B
        // position of the fp32 box (32-byte chunk j / 2 of row r XOR r % 4)
        for (int e0 = lane; e0 < n16; e0 += 32 * 4) {
          uint2 v[4];
#pragma unroll
          for (int u = 0; u < 4; ++u)
            if (e0 + 32 * u < n16) v[u] = lds64(lo + (e0 + 32 * u) * 8);
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int e = e0 + 32 * u;
            if (e < n16) {
              const int r = e >> 3, j = e & 7;
              const float4 f = make_float4(__uint_as_float(v[u].x << 16), __uint_as_float(v[u].x & 0xffff0000u),
                                           __uint_as_float(v[u].y << 16), __uint_as_float(v[u].y & 0xffff0000u));
              tc::sts128(hi + r * 128 + ((((j >> 1) ^ (r & 3)) << 5) | ((j & 1) << 4)), f);
            }
          }
        }
      } else {
        for (int e0 = lane; e0 < n16; e0 += 32 * 4) {
          float4 v[4];
#pragma unroll
          for (int u = 0; u < 4; ++u)
            if (e0 + 32 * u < n16) v[u] = tc::lds128(hi + (e0 + 32 * u) * 16);
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int e = e0 + 32 * u;
            if (e < n16) {
              float4 h, l;
              if (kRawHi) {            // the MMA reads trunc(v) out of the raw box; lo = v - trunc(v) is exact
                h.x = tc::trunc_tf32(v[u].x); h.y = tc::trunc_tf32(v[u].y);
                h.z = tc::trunc_tf32(v[u].z); h.w = tc::trunc_tf32(v[u].w);
                l.x = v[u].x - h.x; l.y = v[u].y - h.y; l.z = v[u].z - h.z; l.w = v[u].w - h.w;
              } else {
                h.x = tc::to_tf32(v[u].x); h.y = tc::to_tf32(v[u].y); h.z = tc::to_tf32(v[u].z); h.w = tc::to_tf32(v[u].w);
                l.x = tc::to_tf32(v[u].x - h.x); l.y = tc::to_tf32(v[u].y - h.y);
                l.z = tc::to_tf32(v[u].z - h.z); l.w = tc::to_tf32(v[u].w - h.w);
                tc::sts128(hi + e * 16, h);
              }
              tc::sts128(lo + e * 16, l);
            }
          }
        }
      }
      tc::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&bars.conv[cw]);
    }
  } else {
    // ------------------------------- epilogue --------------------------------------------------
    // Quadrant q holds output rows 16q..16q+15: their W'hi products on lanes 0-15, W'lo.Zhi on lanes 16-31.
    // TMEM -> registers -> (lo lanes hand their part down by shuffle) -> 128-byte-swizzled staging tile -> one
    // TMA store (or reduce-add) of the [N x 32] box: full 128-byte row segments reach L2, columns beyond K are
    // clipped by the tensor map.
    const int quad = warp & 3;
    const int r = quad * 16 + (lane & 15);                   // output row of this thread
    const bool hi_lane = lane < 16;
    const bool issuer = (quad == 0) && (lane == 0);
    const bool active = quad * 16 < N;                       // warp-uniform
    int ab = 0, ab_phase = 0;
    int ob = 0;
    for (long long t = t_begin; t < t_end; ++t) {
      tc::mbar_wait(&bars.acc_full[ab], ab_phase);
      tc::tc_fence_after();
      float d[32];
      if (active) {
        const uint32_t ta = tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(kTmemAcc0 + ab * kAccCols);
        if (kBf16) {                                                  // W'hi.Zhi  |  W'lo.Zhi  (Zlo = 0)
          tc::tmem_ld_32x32(ta, d);
          tc::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) d[j] = neg2s * (d[j] + __shfl_down_sync(0xffffffffu, d[j], 16));
        } else {
          float e[32];
          tc::tmem_ld_32x32(ta, d);
          tc::tmem_ld_32x32(ta + 32, e);
          tc::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float mine = hi_lane ? d[j] + e[j] : d[j];             // W'hi.(Zhi + Zlo)  |  W'lo.Zhi
            d[j] = neg2s * (mine + __shfl_down_sync(0xffffffffu, mine, 16));
        }
        }
      }
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&bars.acc_empty[ab]); // the accumulator is free as soon as it is in registers
      // the staging buffer `ob` was last read by the TMA store issued two tiles ago
      if (issuer) tc::tma_store_wait_read<1>();
      tc::named_bar_sync(2, kEpiWarps * 32);
      if (active && hi_lane && r < N) {
        if (kBf16) {                      // 64-byte rows, 64-byte swizzle: 16-byte chunk q at q ^ ((r / 2) % 4)
          const uint32_t row = tc::smem_u32(obuf + ob * kObufBytes) + r * 64;
#pragma unroll
          for (int q = 0; q < 4; ++q)
            tc::sts128(row + ((q ^ ((r >> 1) & 3)) << 4),
                       make_float4(__uint_as_float(pack_bf16x2(d[8 * q], d[8 * q + 1])),
                                   __uint_as_float(pack_bf16x2(d[8 * q + 2], d[8 * q + 3])),
                                   __uint_as_float(pack_bf16x2(d[8 * q + 4], d[8 * q + 5])),
                                   __uint_as_float(pack_bf16x2(d[8 * q + 6], d[8 * q + 7]))));
        } else {
          const uint32_t row = tc::smem_u32(obuf + ob * kObufBytes) + r * 128;
#pragma unroll
          for (int j = 0; j < 8; ++j)
            tc::sts128(row + ((j ^ (r & 7)) << 4), make_float4(d[4 * j], d[4 * j + 1], d[4 * j + 2], d[4 * j + 3]));
        }
      }
      tc::fence_proxy_async_smem();
      tc::named_bar_sync(2, kEpiWarps * 32);
      if (issuer) {
        const int col0 = (int)(tile_of(t) * kCols);
        if (accumulate) tc::tma_reduce_add_3d(&tmo, obuf + ob * kObufBytes, col0, 0, p);
        else tc::tma_store_3d(&tmo, obuf + ob * kObufBytes, col0, 0, p);
        tc::tma_store_commit();
      }
      ob ^= 1;
      if (++ab == kAccBufs) { ab = 0; ab_phase ^= 1; }
    }
    if (issuer) tc::tma_store_wait<0>();
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 1) tc::tmem_dealloc(tmem, kTmemCols);
}

__global__ void __launch_bounds__(kThreads, kCtasPerSm)
grad_tc_kernel(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ CUtensorMap tmy,
               const __grid_constant__ CUtensorMap tmo, int Bx, int By, long long K, const float* __restrict__ Wimg,
               int rb, int N, float neg2s, int accumulate, int ctx_period, int ctx_len) {
  grad_tc_body<false>(tmx, tmy, tmo, Bx, By, K, Wimg, rb, N, neg2s, accumulate, ctx_period, ctx_len);
}

// bf16 videos and gradient (see grad_tc_body): same shared memory, registers and tensor memory as grad_tc_kernel
__global__ void __launch_bounds__(kThreads, kCtasPerSm)
grad_tc_bf16_kernel(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ CUtensorMap tmy,
                    const __grid_constant__ CUtensorMap tmo, int Bx, int By, long long K, const float* __restrict__ Wimg,
                    int rb, int N, float neg2s, int accumulate, int ctx_period, int ctx_len) {
  grad_tc_body<true>(tmx, tmy, tmo, Bx, By, K, Wimg, rb, N, neg2s, accumulate, ctx_period, ctx_len);
}

// dynamic shared memory: hi[kStages] | lo[kStages] | 2 output staging tiles | barriers, + 1 KB for the alignment
constexpr size_t grad_smem_bytes(int rows_max) {
  return (size_t)kStages * 2 * rows_max * 128 + 2 * kObufBytes + sizeof(Bars) + 1024;
}
// per SM: 228 KB of shared memory, of which the hardware reserves 1 KB per CTA
static_assert(grad_smem_bytes(kMaxN) + 1024 <= 228 * 1024 / kCtasPerSm, "two CTAs per SM");

}  // namespace

bool tc_grad_supported(const float* x, const float* y, int Bx, int By, long long K, const float* gx, const float* gy) {
  if (Bx % 8 || By % 8 || Bx + By > 128 || Bx > kMaxN || By > kMaxN || Bx < 8 || By < 8) return false;
  if (K % 4 != 0 || K < 128) return false;
  if ((reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(y) & 15)) return false;
  if ((gx && (reinterpret_cast<uintptr_t>(gx) & 15)) || (gy && (reinterpret_cast<uintptr_t>(gy) & 15))) return false;
  return true;
}

// img: the W' images of build_w_image_kernel ([nprob][2][128 x 128] floats); rb = 0: gradient of the x rows, 1: y rows
// bf16: videos and `out` are bf16 (grad_tc_bf16_kernel), no accumulation
static int launch_grad_rows(const CUtensorMap& tmx, const CUtensorMap& tmy, const float* img, int rb, int nprob, int Bx,
                            int By, long long K, float s, void* out, int accumulate, bool bf16, cudaStream_t st) {
  const int N = rb ? By : Bx;
  const size_t smem = grad_smem_bytes(Bx > By ? Bx : By);
  // output [nprob][N][K], box [N x 32]: fp32 with the 128-byte swizzle, bf16 with the 64-byte swizzle (each matches
  // its staging tile)
  CUtensorMap tmo;
  if (int rc = bf16 ? encode_tmap_3d(&tmo, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, CU_TENSOR_MAP_SWIZZLE_64B, out, (uint64_t)K,
                                     (uint64_t)N, (uint64_t)nprob, (uint64_t)K * 2, (uint64_t)K * 2 * N, kBoxCols,
                                     (uint32_t)N)
                    : encode_tmap_3d(&tmo, out, (uint64_t)K, (uint64_t)N, (uint64_t)nprob, (uint64_t)K * 4,
                                     (uint64_t)K * 4 * N, kBoxCols, (uint32_t)N))
    return rc;
  auto kernel = bf16 ? grad_tc_bf16_kernel : grad_tc_kernel;
  static size_t attr_smem[2][kMaxDevices] = {};
  if (smem_attr_needed(attr_smem[bf16 ? 1 : 0], smem)) {
    KCCOT_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // the whole 228 KB as shared memory, so that a second CTA (of this or another kernel) still finds its seat
    KCCOT_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                    (int)cudaSharedmemCarveoutMaxShared));
  }
  long long ntiles = (K + kCols - 1) / kCols;
  // shared-context hint: only the gradient of the y rows (the fake video) skips the context tiles (the skipped
  // columns are left untouched)
  int ctx_period = 0, ctx_len = 0;
  if (rb == 1 && Bx == By && ctx_boxes(K, &ctx_period, &ctx_len))
    ntiles = ntiles / ctx_period * (ctx_period - ctx_len);
  else
    ctx_period = ctx_len = 0;
  const int sms = num_sms();
  int gx = (sms + nprob - 1) / nprob;
  if ((long long)gx * nprob > sms) {
    // several waves of CTAs (more problems than SMs): pick the column split whose last wave wastes the fewest SMs,
    // keeping at least 32 tiles per CTA (256 problems on 148 SMs: 1 range each = 2 waves at 86 %, 4 ranges = 7 at 99 %).
    // A wave counts one CTA per SM although two fit: counting two (8 ranges for 256 problems) was measured 0.15 %
    // slower on config 4.
    int best = gx;
    double best_eff = 0.0;
    for (int g = gx; g <= gx + 7 && (long long)g * 32 <= ntiles; ++g) {
      const long long ctas = (long long)g * nprob, waves = (ctas + sms - 1) / sms;
      const double eff = (double)ctas / (double)(waves * sms);
      if (eff > best_eff + 0.02) { best_eff = eff; best = g; }
    }
    gx = best;
  }
  if (gx > ntiles) gx = (int)ntiles;
  if (gx < 1) gx = 1;
  dim3 grid(gx, nprob);
  KCCOT_CUDA(launch_pdl(kernel, grid, dim3(kThreads), smem, st, tmx, tmy, tmo, Bx, By, K, img, rb, N, -2.f * s,
                        accumulate, ctx_period, ctx_len));
  KCCOT_LAUNCH_CHECK();
  return KCCOT_OK;
}

size_t tc_grad_ws_bytes(int nprob) { return (size_t)nprob * 2 * kImgFloats * sizeof(float); }

template <bool kMixed>
static int launch_grad_common(const float* C, const float* x, const float* y, int nprob, int Bx, int By, long long K,
                              float s, float* gx, float* gy, int accumulate, float* img, cudaStream_t st) {
  if (!gx && !gy) return KCCOT_OK;
  const int rb_first = gx ? 0 : 1, nrb = (gx ? 1 : 0) + (gy ? 1 : 0);
  KCCOT_CUDA(launch_pdl(build_w_image_kernel<kMixed>, dim3(kMaxN, nrb, nprob), dim3(128), 0, st, C, Bx, By, rb_first, img));
  KCCOT_LAUNCH_CHECK();
  CUtensorMap tmx, tmy;
  if (int rc = encode_tmap_3d(&tmx, x, (uint64_t)K, (uint64_t)Bx, (uint64_t)nprob, (uint64_t)K * 4, (uint64_t)K * 4 * Bx,
                              kBoxCols, (uint32_t)Bx, true))
    return rc;
  if (int rc = encode_tmap_3d(&tmy, y, (uint64_t)K, (uint64_t)By, (uint64_t)nprob, (uint64_t)K * 4, (uint64_t)K * 4 * By,
                              kBoxCols, (uint32_t)By, true))
    return rc;
  if (gy)
    if (int rc = launch_grad_rows(tmx, tmy, img, 1, nprob, Bx, By, K, s, gy, accumulate, false, st)) return rc;
  if (gx)
    if (int rc = launch_grad_rows(tmx, tmy, img, 0, nprob, Bx, By, K, s, gx, accumulate, false, st)) return rc;
  return KCCOT_OK;
}

int launch_grad_tc_bf16(const float* Cbar3, const uint16_t* x, const uint16_t* y, int nprob, int B, long long K,
                        float s, uint16_t* gx, uint16_t* gy, float* Wws, cudaStream_t st) {
  if (!gx && !gy) return KCCOT_OK;
  const int rb_first = gx ? 0 : 1, nrb = (gx ? 1 : 0) + (gy ? 1 : 0);
  KCCOT_CUDA(launch_pdl(build_w_image_kernel<true>, dim3(kMaxN, nrb, nprob), dim3(128), 0, st, Cbar3, B, B, rb_first,
                        Wws));
  KCCOT_LAUNCH_CHECK();
  CUtensorMap tmx, tmy;     // [rows x 32] bf16 boxes, unswizzled (the converters place them)
  if (int rc = encode_tmap_3d(&tmx, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, CU_TENSOR_MAP_SWIZZLE_NONE, x, (uint64_t)K,
                              (uint64_t)B, (uint64_t)nprob, (uint64_t)K * 2, (uint64_t)K * 2 * B, kBoxCols, (uint32_t)B))
    return rc;
  if (int rc = encode_tmap_3d(&tmy, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, CU_TENSOR_MAP_SWIZZLE_NONE, y, (uint64_t)K,
                              (uint64_t)B, (uint64_t)nprob, (uint64_t)K * 2, (uint64_t)K * 2 * B, kBoxCols, (uint32_t)B))
    return rc;
  if (gy)
    if (int rc = launch_grad_rows(tmx, tmy, Wws, 1, nprob, B, B, K, s, gy, 0, true, st)) return rc;
  if (gx)
    if (int rc = launch_grad_rows(tmx, tmy, Wws, 0, nprob, B, B, K, s, gx, 0, true, st)) return rc;
  return KCCOT_OK;
}

// Wws: tc_grad_ws_bytes(nprob) of scratch for the W' images
int launch_grad_tc(const float* Cbar3, const float* x, const float* y, int nprob, int Bx, int By, long long K, float s,
                   float* gx, float* gy, int accumulate, float* Wws, cudaStream_t st) {
  return launch_grad_common<true>(Cbar3, x, y, nprob, Bx, By, K, s, gx, gy, accumulate, Wws, st);
}

int launch_grad_pair_tc(const float* Cbar, const float* x, const float* y, int nprob, int Bx, int By, long long K,
                        float s, float* gx, float* gy, int accumulate, float* Wws, cudaStream_t st) {
  return launch_grad_common<false>(Cbar, x, y, nprob, Bx, By, K, s, gx, gy, accumulate, Wws, st);
}

}  // namespace kccot
