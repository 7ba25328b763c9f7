// cd_block.cuh — K1, the per-row coordinate descent of eALS as BLOCKED coordinate descent (all row
// lengths; the plain one-reduction-per-factor form lives in cd_sweep.cuh for comparison).
//
// Same arithmetic as MF_fastALS::update_user_thread / update_item_thread (MF_fastALS.cpp:243-322,
// 338-407), reorganised so that a row needs ONE team-wide reduction per block of 16 factors instead
// of one per factor.  For a block B = {f0..f0+15} of the row x, with the prediction cache p_j
// (current <x, y_j>) at the start of the block:
//
//   z_j  = w_j r_j - c_j p_j                        c_j = w_j - Wi[item]
//   P_f  = sum_j z_j y_jf                           (f in B)
//   G_kf = sum_j c_j y_jk y_jf                      (k, f in B; the row's local 16 x 16 Gram)
//   t_f  = sum_k x_k S[f][k]                        (all K, x at the start of the block)
//   H_kf = G_kf + g S[k][f]                         g = 1 (user side) | Wi[row] (item side)
//
// the reference's sequential updates inside the block are, exactly,
//
//   for f in B (ascending):  numer = P_f - g t_f + x_f H_ff - sum_{k in B, k < f} d_k H_kf
//                            x_f'  = numer / (H_ff + reg) ;  d_f = x_f' - x_f
//
// (substitute p_j(current) = p_j + sum_{k<f} d_k y_jk into :297-305 and collect terms), followed by
// p_j += sum_{f in B} d_f y_jf.  Only the floating-point summation order differs.
//
// G is GEMM-shaped (16 x n times n x 16) and goes to the fp64 tensor cores (mma.sync.m8n8k4.f64, three
// 8 x 8 tiles — only the lower triangle of the symmetric system is needed); P rides along as two more
// tiles (z in column 0 of the B operand); the prediction-cache update and the 16-step solve are plain
// fp64.  On B200 a DMMA costs exactly 8 DFMAs of the one fp64 pipe (tests/micro/fp64_rate.cu).
//
// Data movement: the 128-byte line [f0, f0+16) of every gathered row is copied global -> shared with
// cp.async (16 B per lane, 8 lanes per line: whole lines, no register staging), XOR-swizzled in
// 16-byte chunks so that both the per-nonzero row reads (LDS.128) and the tensor-core fragment reads
// are conflict-free.  (TMA tile::gather4 writes the same layout and was measured: not faster here,
// DESIGN.md §3.1.)
//
// Three drivers share the device code (bucket limits in eals_b200.cu):
//   * cd_warp_block_kernel — one WARP per row of 1..128 nonzeros (1..4 per lane), persistent CTAs, the
//                            other side's S cache resident in shared memory, no CTA barrier per row.
//   * cd_row_block_kernel  — one CTA per row of 129..512 nonzeros (4 warps x 2 or 3, 8 warps x 2 nonzeros
//                            per thread), everything on chip.
//   * heavy_* kernels      — rows of any length split into slabs of 128 nonzeros; per block one launch
//                            for the slab partials (+ the deferred cache update of the previous block),
//                            one for the grouped reduction and one for the per-row solve; prediction
//                            cache in HBM; slabs launched in neighbour order for L2 reuse.
#pragma once

#include "cd_sweep.cuh"
#include "common.cuh"

namespace eals {

constexpr int kBlkThreads = 256;
constexpr int kBlkWarps = kBlkThreads / 32;
constexpr int kPartLen = 208;   // 3 tiles x 32 lanes x 2 (C fragments) + 16 (P)
constexpr int kMaxSlab = 256;   // nonzeros per slab of a heavy row (one per thread): 128 or 256, chosen by the host

// ---- swizzled tile: row r = 128 bytes, 16-byte chunk c stored at chunk position c ^ (r & 7) ----
__device__ __forceinline__ uint32_t tile_chunk_off(int r, int c) { return (uint32_t)(r * 128 + (((c ^ r) & 7) << 4)); }
__device__ __forceinline__ double tile_elem(const unsigned char* tile, int r, int e) {
  return *reinterpret_cast<const double*>(tile + tile_chunk_off(r, e >> 1) + ((e & 1) << 3));
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src, int src_bytes) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(gmem_src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// Stage factor block fb of n gathered rows into the tile; rows [n, n_pad) are zero-filled.  The source
// comes from a table of row base pointers (rowp_s[r] = &Y[idx[r]][0]) built once per row: per 16-byte
// chunk one LDS.64, one add and the cp.async.  Thread t always copies chunk column t & 7 of rows
// (t >> 3), (t >> 3) + nthreads/8, ...  (r01e: the index arithmetic of the version above was 16.5 % of
// the team kernel's instructions.)
__device__ __forceinline__ void stage_tile_rows(unsigned char* tile, const double* const* rowp_s, int n, int n_pad,
                                                int fb, int tid, int nthreads) {
  const int c = tid & 7;
  const uint32_t col_bytes = (uint32_t)(fb * (kFB * 8) + c * 16);
  for (int r = tid >> 3; r < n_pad; r += nthreads >> 3) {
    const bool live = r < n;
    const unsigned char* src = reinterpret_cast<const unsigned char*>(rowp_s[live ? r : 0]) + col_bytes;
    cp_async16(tile + (uint32_t)(r * 128) + (uint32_t)(((c ^ r) & 7) << 4), src, live ? 16 : 0);
  }
}

// Blocks fb - 1 and fb of the same rows into two tiles with ONE pass over the row-pointer table
// (heavy_step: the deferred cache update and the Gram pass need consecutive blocks of the same rows).
__device__ __forceinline__ void stage_two_tiles(unsigned char* tile_prev, unsigned char* tile, const double* const* rowp_s,
                                                int n, int n_pad, int fb, bool do_prev, bool do_cur, int tid, int nthreads) {
  const int c = tid & 7;
  const uint32_t col_bytes = (uint32_t)(fb * (kFB * 8) + c * 16);
  for (int r = tid >> 3; r < n_pad; r += nthreads >> 3) {
    const bool live = r < n;
    const unsigned char* src = reinterpret_cast<const unsigned char*>(rowp_s[live ? r : 0]) + col_bytes;
    const uint32_t dst = (uint32_t)(r * 128) + (uint32_t)(((c ^ r) & 7) << 4);
    if (do_prev) cp_async16(tile_prev + dst, src - kFB * 8, live ? 16 : 0);
    if (do_cur) cp_async16(tile + dst, src, live ? 16 : 0);
  }
}

__device__ __forceinline__ void dmma_884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// Load the 16 doubles of tile row r into registers.
__device__ __forceinline__ void load_tile_row(const unsigned char* tile, int r, double (&y)[16]) {
#pragma unroll
  for (int c = 0; c < 8; c++) {
    const double2 d = *reinterpret_cast<const double2*>(tile + tile_chunk_off(r, c));
    y[2 * c] = d.x;
    y[2 * c + 1] = d.y;
  }
}

// ---------------------------------------------------------------------------------------------
// One WARP per row, 1 .. 32*MAXM nonzeros (lane l owns nonzeros l, l+32, ...), PERSISTENT CTAs.
//
// Measured on the first blocked version (profiles/README.md r01c): 39 % of the stall samples sat on
// the S-cache loads of the per-block solve (K x K fp64 = 128 KB at K = 128 does not stay in L1) and
// 9 % of the instructions were the selects of the 16-value shuffle reduction.  Hence:
//   * the whole S cache is copied to shared memory ONCE per CTA (LD <= 128; CTAs are persistent and
//     stride over the rows), every S access of the solve is an LDS;
//   * the right-hand side P_f = sum_j z_j y_jf rides on the tensor cores as two more 8 x 8 tiles (z in
//     column 0 of the B operand) — no cross-lane reduction at all;
//   * S.x is split over FACTOR lanes (lane = (f, half of k); S is symmetric, so the lane walks a
//     column of S with unit stride across lanes) — one shuffle instead of a 16-value butterfly;
//   * the 16-step in-block Gauss-Seidel is multiply/shuffle/fma only (one reciprocal per factor,
//     taken in parallel before the loop).
// ---------------------------------------------------------------------------------------------
// S in shared memory: symmetric, so only the 16 x 16 blocks on and below the block diagonal are
// kept (LD = 128: 36 blocks, 78 KB instead of 128 KB — the difference buys 50 % more resident
// row-warps per SM).  Block (bi, bj), bi >= bj, holds S[16 bi + r][16 bj + c] at [r * 17 + c]; the odd
// row stride makes both the row walk (element of the block's transpose) and the column walk
// conflict-free across the 16 factor lanes.
constexpr int kSBlk = 16 * 17;
// The 16 x 16 block system H of one row, lower triangle only, row stride 17: the fragment lanes store
// their 8 x 8 tiles (T00, T10, T11) as they hold them and solve lane f reads ROW f (H is symmetric and
// step f only needs H[f][s], s <= f) — conflict-free.  The first layout (stride 16 plus a transposed copy
// of T10 for column reads) made every store an 8-way bank conflict: ~100 of the 455 shared-memory
// wavefronts per row and block of the short-row kernel, which is shared-memory bound (profiles r01h).
constexpr int kGsStride = 17;
constexpr int kGsLen = 16 * kGsStride;
__host__ __device__ constexpr int s_tri(int bi, int bj) { return bi * (bi + 1) / 2 + bj; }

template <int LD, int MAXM>
struct WarpBlockSmem {
  static constexpr bool kSInSmem = LD <= 128;
  static constexpr int kNB = LD / 16;
  static constexpr int kRows = 32 * MAXM;
  static constexpr size_t kS = kSInSmem ? (size_t)s_tri(kNB, 0) * kSBlk * 8 : 0;
  static constexpr size_t kTile = (size_t)kRows * 128;
  // tile | row pointers | x | Gs | Pt[16] | delta[16]
  static constexpr size_t kBytesPerWarp = kTile + (size_t)kRows * 8 + (size_t)LD * 8 + (kGsLen + 16 + 16) * 8;
  static constexpr int kMaxWarps = MAXM == 1 ? 16 : (MAXM == 2 ? 12 : (MAXM == 3 ? 9 : 7));
};

// Gram + right-hand-side fragments of tile rows [0, r1): frag[0..5] as gram_fragments, frag[6..7] =
// P rows 0..7, frag[8..9] = P rows 8..15 (column 0 of each tile holds the sums).
__device__ __forceinline__ void gram_rhs_fragments(const unsigned char* tile, const double* c_s, const double* z_s,
                                                   int r0, int r1, double (&frag)[10]) {
  const int lane = lane_id();
  const int rr = lane & 3, e0 = lane >> 2;
  const uint32_t off_lo = (uint32_t)(rr * 128 + ((e0 & 1) << 3));
  for (int j0 = r0; j0 < r1; j0 += 4) {
    const int r = j0 + rr;
    const uint32_t sw = (uint32_t)(r & 7);
    const unsigned char* rowp = tile + (size_t)j0 * 128 + off_lo;
    const double a0 = *reinterpret_cast<const double*>(rowp + ((((uint32_t)(e0 >> 1)) ^ sw) << 4));
    const double a1 = *reinterpret_cast<const double*>(rowp + ((((uint32_t)(4 + (e0 >> 1))) ^ sw) << 4));
    const double cj = c_s[r];
    const double zj = e0 == 0 ? z_s[r] : 0.0;
    const double b0 = cj * a0, b1 = cj * a1;
    dmma_884(frag[0], frag[1], a0, b0);
    dmma_884(frag[2], frag[3], a1, b0);
    dmma_884(frag[4], frag[5], a1, b1);
    dmma_884(frag[6], frag[7], a0, zj);
    dmma_884(frag[8], frag[9], a1, zj);
  }
}

// The same for tile rows [r0, r0 + 32) with c_j / z_j taken from the owning lanes' registers (row
// r0 + l belongs to lane l of this warp): one shuffle each instead of a shared-memory array — the
// warp-per-row kernels spend their shared memory on tiles (= rows in flight), not on scalars.
__device__ __forceinline__ void gram_rhs_fragments_reg(const unsigned char* tile, double c_lane, double z_lane,
                                                       int r0, int r1, double (&frag)[10]) {
  const int lane = lane_id();
  const int rr = lane & 3, e0 = lane >> 2;
  const uint32_t off_lo = (uint32_t)(rr * 128 + ((e0 & 1) << 3));
  for (int j0 = r0; j0 < r1; j0 += 4) {
    const int r = j0 + rr;
    const uint32_t sw = (uint32_t)(r & 7);
    const unsigned char* rowp = tile + (size_t)j0 * 128 + off_lo;
    const double a0 = *reinterpret_cast<const double*>(rowp + ((((uint32_t)(e0 >> 1)) ^ sw) << 4));
    const double a1 = *reinterpret_cast<const double*>(rowp + ((((uint32_t)(4 + (e0 >> 1))) ^ sw) << 4));
    const double cj = __shfl_sync(kFullMask, c_lane, (j0 - r0) + rr);
    const double zq = __shfl_sync(kFullMask, z_lane, (j0 - r0) + rr);
    const double zj = e0 == 0 ? zq : 0.0;
    const double b0 = cj * a0, b1 = cj * a1;
    dmma_884(frag[0], frag[1], a0, b0);
    dmma_884(frag[2], frag[3], a1, b0);
    dmma_884(frag[4], frag[5], a1, b1);
    dmma_884(frag[6], frag[7], a0, zj);
    dmma_884(frag[8], frag[9], a1, zj);
  }
}

template <int LD, int MAXM, bool USER>
__global__ void __launch_bounds__(WarpBlockSmem<LD, MAXM>::kMaxWarps * 32, 1)
cd_warp_block_kernel(CdSide a, const int32_t* __restrict__ order, int first, int count) {
  extern __shared__ __align__(128) unsigned char smem[];
  using Sm = WarpBlockSmem<LD, MAXM>;
  const int warp = threadIdx.x >> 5, lane = lane_id();
  const int wpb = blockDim.x >> 5;

  // the S cache of the other side, resident in shared memory for the CTA's lifetime
  const double* S_s = reinterpret_cast<const double*>(smem);
  if (Sm::kSInSmem) {
    double* S_w = reinterpret_cast<double*>(smem);
    for (int t = threadIdx.x; t < s_tri(Sm::kNB, 0) * 256; t += blockDim.x) {
      const int blk = t >> 8, r = (t >> 4) & 15, c = t & 15;
      int bi = 0;
      while (s_tri(bi + 1, 0) <= blk) bi++;
      const int bj = blk - s_tri(bi, 0);
      S_w[blk * kSBlk + r * 17 + c] = __ldg(a.S + (size_t)(bi * 16 + r) * LD + bj * 16 + c);
    }
    __syncthreads();
  }

  unsigned char* base = smem + Sm::kS + (size_t)warp * Sm::kBytesPerWarp;
  unsigned char* tile = base;
  const double** rowp_s = reinterpret_cast<const double**>(base + Sm::kTile);
  double* x_s = reinterpret_cast<double*>(base + Sm::kTile + (size_t)Sm::kRows * 8);
  double* Gs = x_s + LD;
  double* Pt = Gs + kGsLen;
  double* delta_s = Pt + 16;

  const int K = a.K;
  const int nblocks = (K + kFB - 1) / kFB;
  const int f = lane & 15, hh = lane >> 4;

  // Descriptor of the NEXT row, fetched in four dependent steps (order -> offsets -> indices ->
  // weights) spread over the factor blocks of the current row: measured on rows of 65..128 nonzeros
  // (profiles r01g) a warp spent ~15 % of its time stalled on exactly this chain at every row start.
  constexpr int XN = (LD + 31) / 32;
  const int stride = gridDim.x * wpb;
  int row_n = 0, n_n = 0, id_n[MAXM];
  int64_t p0_n = 0, p1_n = 0;
  double wi_n[MAXM], pc_n[MAXM], wi_row_n = 0.0, x_n[XN];
  uint32_t g_n[MAXM];
#pragma unroll
  for (int m = 0; m < MAXM; m++) { id_n[m] = 0; wi_n[m] = 0.0; pc_n[m] = 0.0; g_n[m] = 0; }
#pragma unroll
  for (int i = 0; i < XN; i++) x_n[i] = 0.0;
  auto fetch_next = [&](int stage, int slot_n) {
    if (slot_n >= count) return;
    if (stage == 0) {
      row_n = order[first + slot_n];
    } else if (stage == 1) {
      p0_n = a.ptr[row_n];
      p1_n = a.ptr[row_n + 1];
      const double* xr = a.X + (size_t)(a.row_base + row_n) * LD;
#pragma unroll
      for (int i = 0; i < XN; i++)
        if (lane + 32 * i < LD) x_n[i] = xr[lane + 32 * i];
      if (!USER) wi_row_n = a.Wi[a.row_base + row_n];
    } else if (stage == 2) {
      n_n = (int)(p1_n - p0_n);
#pragma unroll
      for (int m = 0; m < MAXM; m++) {
        const int j = m * 32 + lane;
        if (j < n_n) {
          id_n[m] = a.idx[p0_n + j];
          if (a.use_cache) pc_n[m] = a.pc_in[p0_n + j];
          if (a.pc_out) g_n[m] = a.pc_map[p0_n + j];
        }
      }
    } else if (USER) {
#pragma unroll
      for (int m = 0; m < MAXM; m++)
        if (m * 32 + lane < n_n) wi_n[m] = a.Wi[id_n[m]];
    }
  };
  {
    const int slot0 = blockIdx.x * wpb + warp;
#pragma unroll
    for (int st = 0; st < 4; st++) fetch_next(st, slot0);
  }

  for (int slot = blockIdx.x * wpb + warp; slot < count; slot += stride) {
    const int row = row_n;
    const int64_t p0 = p0_n;
    const int n = n_n;
    const int n_pad = (n + 3) & ~3;
    const int grow = a.row_base + row;
    const double wi_row = USER ? 0.0 : wi_row_n;
    const double g = USER ? 1.0 : wi_row;

    double pr[MAXM], cw[MAXM], wr[MAXM];
    uint32_t gpos[MAXM];
#pragma unroll
    for (int m = 0; m < MAXM; m++) {
      const int j = m * 32 + lane;
      pr[m] = 0.0; cw[m] = 0.0; wr[m] = 0.0;
      gpos[m] = g_n[m];
      if (j < n) {
        rowp_s[j] = a.Y + (size_t)id_n[m] * LD;
        const double w = a.val ? a.val[p0 + j] : 1.0;
        wr[m] = w * w;
        cw[m] = w - (USER ? wi_n[m] : wi_row);
        if (a.use_cache) pr[m] = pc_n[m];
      }
    }
#pragma unroll
    for (int i = 0; i < XN; i++)
      if (lane + 32 * i < LD) x_s[lane + 32 * i] = x_n[i];
    __syncwarp();
    const int stages_in_loop = nblocks < 4 ? nblocks : 4;

    if (!a.use_cache) {
      // Prediction cache from scratch, p_j = <x, y_j> (MF_fastALS.cpp:261-270): straight from global
      // memory, 8 lanes per nonzero (16 bytes each of every 128-byte line of the gathered row), four
      // nonzeros per step and every load independent — instead of staging block after block with a full
      // memory round trip each (first sweep after setTrain: +60 ms on c4 before).
      double* ptmp = reinterpret_cast<double*>(tile);   // the tile is free here
      const int g8 = lane >> 3, gl = lane & 7;
#pragma unroll 2
      for (int j0 = 0; j0 < n; j0 += 4) {
        const int j = j0 + g8;
        double acc0 = 0.0, acc1 = 0.0;
        if (j < n) {
          const double* yrow = rowp_s[j];
#pragma unroll
          for (int c = 0; c < LD; c += kFB) {
            const double2 d = ldg2(yrow + c + gl * 2);
            acc0 += x_s[c + gl * 2] * d.x;
            acc1 += x_s[c + gl * 2 + 1] * d.y;
          }
        }
        double acc = acc0 + acc1;
        acc += __shfl_xor_sync(kFullMask, acc, 1);
        acc += __shfl_xor_sync(kFullMask, acc, 2);
        acc += __shfl_xor_sync(kFullMask, acc, 4);
        if (j < n && gl == 0) ptmp[j] = acc;
      }
      __syncwarp();
#pragma unroll
      for (int m = 0; m < MAXM; m++)
        if (m * 32 + lane < n) pr[m] = ptmp[m * 32 + lane];
      __syncwarp();
    }

    stage_tile_rows(tile, rowp_s, n, n_pad, 0, lane, 32);
    cp_async_commit();
    for (int fb = 0; fb < nblocks; fb++) {
      const int f0 = fb * kFB;
      if (fb < 4) fetch_next(fb, slot + stride);
      // S.x for this block while the tile is in flight: t_f = sum_k x_k S[k][f0+f]; lane = (f, half
      // of the k blocks)
      double tsum;
      if (Sm::kSInSmem) {
        double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 0.0;   // four independent chains
        const int kb0 = (Sm::kNB * hh) / 2, kb1 = (Sm::kNB * (hh + 1)) / 2;
        for (int kb = kb0; kb < kb1; kb++) {
          const double* __restrict__ xk = x_s + kb * 16;
          if (kb <= fb) {   // S[f0+f][16 kb + kk]: row f of block (fb, kb)
            const double* __restrict__ sb = S_s + s_tri(fb, kb) * kSBlk + f * 17;
#pragma unroll
            for (int kk = 0; kk < 16; kk += 4) {
              const double2 xa = *reinterpret_cast<const double2*>(xk + kk);
              const double2 xb = *reinterpret_cast<const double2*>(xk + kk + 2);
              t0 += xa.x * sb[kk];
              t1 += xa.y * sb[kk + 1];
              t2 += xb.x * sb[kk + 2];
              t3 += xb.y * sb[kk + 3];
            }
          } else {          // S[16 kb + kk][f0+f]: column f of block (kb, fb)
            const double* __restrict__ sb = S_s + s_tri(kb, fb) * kSBlk + f;
#pragma unroll
            for (int kk = 0; kk < 16; kk += 4) {
              const double2 xa = *reinterpret_cast<const double2*>(xk + kk);
              const double2 xb = *reinterpret_cast<const double2*>(xk + kk + 2);
              t0 += xa.x * sb[kk * 17];
              t1 += xa.y * sb[(kk + 1) * 17];
              t2 += xb.x * sb[(kk + 2) * 17];
              t3 += xb.y * sb[(kk + 3) * 17];
            }
          }
        }
        tsum = (t0 + t1) + (t2 + t3);
        tsum += __shfl_xor_sync(kFullMask, tsum, 16);
      } else {
        const double* __restrict__ Sc = a.S + (size_t)(hh * (LD / 2)) * LD + f0 + f;
        const double* __restrict__ xh = x_s + hh * (LD / 2);
        double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 0.0;
#pragma unroll 2
        for (int k = 0; k < LD / 2; k += 4) {
          const double2 xa = *reinterpret_cast<const double2*>(xh + k);
          const double2 xb = *reinterpret_cast<const double2*>(xh + k + 2);
          t0 += xa.x * __ldg(Sc + (size_t)k * LD);
          t1 += xa.y * __ldg(Sc + (size_t)(k + 1) * LD);
          t2 += xb.x * __ldg(Sc + (size_t)(k + 2) * LD);
          t3 += xb.y * __ldg(Sc + (size_t)(k + 3) * LD);
        }
        tsum = (t0 + t1) + (t2 + t3);
        tsum += __shfl_xor_sync(kFullMask, tsum, 16);
      }
      cp_async_wait<0>();
      __syncwarp();

      double frag[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
      for (int m = 0; m < MAXM; m++)   // z_j = w_j r_j - c_j p_j; rows beyond n have c = z = 0
        gram_rhs_fragments_reg(tile, cw[m], wr[m] - cw[m] * pr[m], m * 32, min(m * 32 + 32, n_pad), frag);
      // H = G + g S_BB, full symmetric 16 x 16, and P
#pragma unroll
      for (int t = 0; t < 3; t++) {
#pragma unroll
        for (int ii = 0; ii < 2; ii++) {
          int rw = lane >> 2, cl = 2 * (lane & 3) + ii;
          if (t >= 1) rw += 8;
          if (t == 2) cl += 8;
          const double sbb = Sm::kSInSmem ? S_s[s_tri(fb, fb) * kSBlk + rw * 17 + cl]
                                          : __ldg(a.S + (size_t)(f0 + rw) * LD + f0 + cl);
          const double v = frag[2 * t + ii] + g * sbb;
          Gs[rw * kGsStride + cl] = v;
        }
      }
      if ((lane & 3) == 0) {
        Pt[lane >> 2] = frag[6];
        Pt[8 + (lane >> 2)] = frag[8];
      }
      __syncwarp();

      // in-block Gauss-Seidel, lane f (both half-warps compute the same thing)
      double h[16];
#pragma unroll
      for (int k = 0; k < 16; k++) h[k] = Gs[f * kGsStride + k];   // row f = column f (only k < f is used)
      const double hff = Gs[f * kGsStride + f];
      const double xf = x_s[f0 + f];
      double numer = Pt[f] - g * tsum + xf * hff;
      const double rden = 1.0 / (hff + a.reg);
#pragma unroll
      for (int s = 0; s < 16; s++) {
        const double d = numer * rden - xf;
        const double ds = __shfl_sync(kFullMask, d, s);
        if (f > s) numer -= ds * h[s];
      }
      const double xnew = numer * rden;
      if (lane < 16) {
        const bool livef = f0 + f < K;
        if (livef) x_s[f0 + f] = xnew;
        delta_s[f] = livef ? xnew - xf : 0.0;
      }
      __syncwarp();

      double d[16];
#pragma unroll
      for (int e = 0; e < 16; e++) d[e] = delta_s[e];
#pragma unroll
      for (int m = 0; m < MAXM; m++) {
        const int j = m * 32 + lane;
        if (j < n) {
          double y[16];
          load_tile_row(tile, j, y);
          double a0 = pr[m], a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll
          for (int e = 0; e < 16; e += 4) {
            a0 += d[e] * y[e];
            a1 += d[e + 1] * y[e + 1];
            a2 += d[e + 2] * y[e + 2];
            a3 += d[e + 3] * y[e + 3];
          }
          pr[m] = (a0 + a1) + (a2 + a3);
        }
      }
      __syncwarp();
      if (fb + 1 < nblocks) {
        stage_tile_rows(tile, rowp_s, n, n_pad, fb + 1, lane, 32);
        cp_async_commit();
      }
    }
    for (int k = lane; k < K; k += 32) store_row_value(a, (size_t)grow * LD + k, x_s[k]);
    if (a.pc_out) {
#pragma unroll
      for (int m = 0; m < MAXM; m++) {
        const int j = m * 32 + lane;
        if (j < n) pc_emit(a, gpos[m], pr[m]);
      }
    }
    for (int st = stages_in_loop; st < 4; st++) fetch_next(st, slot + stride);   // K < 64: finish the chain here
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------
// One CTA (a team of TW warps) per row of up to 32*TW*MW nonzeros, MW nonzeros per thread: thread t
// owns nonzeros t, t+32*TW, ...; warp w feeds tile rows [w*32*MW, (w+1)*32*MW) to the tensor cores
// (Gram + right-hand side, 5 tiles per 4 nonzeros).  The S.x term of the block is spread over ALL
// threads (thread = (factor, 1/16th of k)) and issued before the wait on the tile, so its loads
// overlap the gather; warp 0 then only runs the 16-step multiply/shuffle/fma recurrence.
// Used as <4, 2> for rows of 129..256 nonzeros (4 CTAs = 4 rows in flight per SM) and <8, 2> for
// 257..512 (2 per SM).  What matters most is the number of ROWS in flight per SM, not the number of
// warps per row: measured on c4, 129..256 as 8 warps x 1 nonzero (2 rows/SM, even with the next
// tile prefetched under the solve) took 73 ms, as 4 warps x 2 nonzeros (4 rows/SM) 62 ms
// (profiles/README.md r01i).  First version (r01b): 143 registers -> 1 CTA/SM, barrier stall 7.8 per
// issue while warp 0 did the whole solve incl. 64 S loads per lane; now capped at 128 registers.
// ---------------------------------------------------------------------------------------------
template <int LD, int TW, int MW>
struct RowBlockSmem {
  static constexpr int kT = TW * 32;                         // threads per CTA (team of TW warps)
  static constexpr int kRows = kT * MW;
  static constexpr size_t kTile = (size_t)kRows * 128;
  static constexpr size_t kIdx = (size_t)kRows * 8;           // row base pointers
  static constexpr size_t kCZ = (size_t)kRows * 16;           // c and z
  static constexpr size_t kX = (size_t)LD * 8;
  static constexpr size_t kSlots = (size_t)TW * kPartLen * 8;
  static constexpr size_t kSmall = (kGsLen + 16 + 16 + 16 + 16 * 16) * 8;   // Gs, Pt, Tt, delta, tpart[<=16][16]
  static constexpr size_t kBytes = kTile + kIdx + kCZ + kX + kSlots + kSmall;
};

template <int LD, int TW, int MW, bool USER>
__global__ void __launch_bounds__(TW * 32, 16 / TW)
cd_row_block_kernel(CdSide a, const int32_t* __restrict__ order, int first) {
  extern __shared__ __align__(128) unsigned char smem[];
  using Sm = RowBlockSmem<LD, TW, MW>;
  constexpr int kT = TW * 32;
  constexpr int kParts = kT / 16;                            // S.x: threads = (factor, part of the k range)
  static_assert(kPartLen + 16 <= kT || TW < 8, "reduction threads");
  unsigned char* tile = smem;
  const double** rowp_s = reinterpret_cast<const double**>(smem + Sm::kTile);
  double* c_s = reinterpret_cast<double*>(smem + Sm::kTile + Sm::kIdx);
  double* z_s = c_s + Sm::kRows;
  double* x_s = z_s + Sm::kRows;
  double* slots = x_s + LD;
  double* Gs = slots + TW * kPartLen;
  double* Pt = Gs + kGsLen;
  double* Tt = Pt + 16;
  double* delta_s = Tt + 16;
  double* tpart = delta_s + 16;    // [kParts][16 factors]

  const int tid = threadIdx.x, lane = lane_id(), warp = tid >> 5;
  const int row = order[first + blockIdx.x];
  const int64_t p0 = a.ptr[row];
  const int n = (int)(a.ptr[row + 1] - p0);
  const int n_pad = (n + 3) & ~3;
  const int grow = a.row_base + row;
  double* xrow = a.X + (size_t)grow * LD;
  const int K = a.K;
  const double wi_row = USER ? 0.0 : a.Wi[grow];
  const double g = USER ? 1.0 : wi_row;

  double pr[MW], cw[MW], wr[MW];
#pragma unroll
  for (int m = 0; m < MW; m++) {
    const int j = m * kT + tid;
    pr[m] = 0.0; cw[m] = 0.0; wr[m] = 0.0;
    if (j < n) {
      const int id = a.idx[p0 + j];
      rowp_s[j] = a.Y + (size_t)id * LD;
      const double w = a.val ? a.val[p0 + j] : 1.0;
      wr[m] = w * w;
      cw[m] = w - (USER ? a.Wi[id] : wi_row);
      if (a.use_cache) pr[m] = a.pc_in[p0 + j];
    }
    c_s[j] = cw[m];
    z_s[j] = 0.0;
  }
  for (int k = tid; k < LD; k += kT) x_s[k] = xrow[k];
  __syncthreads();

  const int nblocks = (K + kFB - 1) / kFB;

  // Pass 1: prediction cache p_j = <x, y_j> (skipped when the symmetric cache is valid): straight from
  // global memory, 8 lanes per nonzero, all loads independent (see cd_warp_block_kernel)
  if (!a.use_cache) {
    const int g8 = tid >> 3, gl = tid & 7;
    for (int j0 = 0; j0 < n; j0 += kT / 8) {
      const int j = j0 + g8;
      double acc0 = 0.0, acc1 = 0.0;
      if (j < n) {
        const double* yrow = rowp_s[j];
#pragma unroll
        for (int c = 0; c < LD; c += kFB) {
          const double2 d = ldg2(yrow + c + gl * 2);
          acc0 += x_s[c + gl * 2] * d.x;
          acc1 += x_s[c + gl * 2 + 1] * d.y;
        }
      }
      double acc = acc0 + acc1;
      acc += __shfl_xor_sync(kFullMask, acc, 1);
      acc += __shfl_xor_sync(kFullMask, acc, 2);
      acc += __shfl_xor_sync(kFullMask, acc, 4);
      if (j < n && gl == 0) z_s[j] = acc;
    }
    __syncthreads();
#pragma unroll
    for (int m = 0; m < MW; m++)
      if (m * kT + tid < n) pr[m] = z_s[m * kT + tid];
    __syncthreads();
  }

  // Pass 2: one blocked update per 16 factors
  const int w_r1 = min((warp + 1) * 32 * MW, n_pad);
  const int tf = tid & 15, tpart_id = tid >> 4;          // S.x: factor and 1/16th of the k range
  constexpr int kPer = LD / kParts;                       // k's per thread
  stage_tile_rows(tile, rowp_s, n, n_pad, 0, tid, kT);
  cp_async_commit();
  for (int fb = 0; fb < nblocks; fb++) {
    const int f0 = fb * kFB;
#pragma unroll
    for (int m = 0; m < MW; m++) {
      const int j = m * kT + tid;
      if (j < n) z_s[j] = wr[m] - cw[m] * pr[m];
    }
    {   // partial t_f = sum over this thread's k's of x_k S[k][f0+f] (S symmetric: unit stride over f)
      const double* __restrict__ Sc = a.S + (size_t)(tpart_id * kPer) * LD + f0 + tf;
      double t0 = 0.0, t1 = 0.0;
#pragma unroll 8
      for (int k = 0; k < kPer; k += 2) {
        t0 += x_s[tpart_id * kPer + k] * __ldg(Sc + (size_t)k * LD);
        if (kPer > 1) t1 += x_s[tpart_id * kPer + k + 1] * __ldg(Sc + (size_t)(k + 1) * LD);
      }
      tpart[tpart_id * 16 + tf] = t0 + t1;
    }
    cp_async_wait<0>();
    __syncthreads();

    double frag[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    gram_rhs_fragments(tile, c_s, z_s, warp * 32 * MW, w_r1, frag);
    double* slot = slots + warp * kPartLen;
#pragma unroll
    for (int t = 0; t < 3; t++) {
      slot[t * 64 + lane * 2] = frag[2 * t];
      slot[t * 64 + lane * 2 + 1] = frag[2 * t + 1];
    }
    if ((lane & 3) == 0) {
      slot[192 + (lane >> 2)] = frag[6];
      slot[200 + (lane >> 2)] = frag[8];
    }
    __syncthreads();
    for (int i = tid; i < kPartLen + 16; i += kT) {
      if (i < kPartLen) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < TW; w++) s += slots[w * kPartLen + i];
        if (i < 192) {   // H = G + g S_BB
          const int t = i >> 6, l = (i & 63) >> 1, ii = i & 1;
          int rw = l >> 2, cl = 2 * (l & 3) + ii;
          if (t >= 1) rw += 8;
          if (t == 2) cl += 8;
          s += g * __ldg(a.S + (size_t)(f0 + rw) * LD + f0 + cl);
          Gs[rw * kGsStride + cl] = s;
        } else {
          Pt[i - 192] = s;
        }
      } else {
        const int ff = i - kPartLen;
        double s = 0.0;
#pragma unroll
        for (int q = 0; q < kParts; q++) s += tpart[q * 16 + ff];
        Tt[ff] = s;
      }
    }
    __syncthreads();
    if (warp == 0) {
      const int ff = lane & 15;
      double h[16];
#pragma unroll
      for (int k = 0; k < 16; k++) h[k] = Gs[ff * kGsStride + k];
      const double hff = Gs[ff * kGsStride + ff];
      const double xf = x_s[f0 + ff];
      double numer = Pt[ff] - g * Tt[ff] + xf * hff;
      const double rden = 1.0 / (hff + a.reg);
#pragma unroll
      for (int sidx = 0; sidx < 16; sidx++) {
        const double d = numer * rden - xf;
        const double ds = __shfl_sync(kFullMask, d, sidx);
        if (ff > sidx) numer -= ds * h[sidx];
      }
      const double xnew = numer * rden;
      if (lane < 16) {
        const bool livef = f0 + ff < K;
        if (livef) x_s[f0 + ff] = xnew;
        delta_s[ff] = livef ? xnew - xf : 0.0;
      }
    }
    __syncthreads();
    {
      double d[16];
#pragma unroll
      for (int e = 0; e < 16; e++) d[e] = delta_s[e];
#pragma unroll
      for (int m = 0; m < MW; m++) {
        const int j = m * kT + tid;
        if (j < n) {
          double y[16];
          load_tile_row(tile, j, y);
          double a0 = pr[m], a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll
          for (int e = 0; e < 16; e += 4) {
            a0 += d[e] * y[e];
            a1 += d[e + 1] * y[e + 1];
            a2 += d[e + 2] * y[e + 2];
            a3 += d[e + 3] * y[e + 3];
          }
          pr[m] = (a0 + a1) + (a2 + a3);
        }
      }
    }
    __syncthreads();
    if (fb + 1 < nblocks) {
      stage_tile_rows(tile, rowp_s, n, n_pad, fb + 1, tid, kT);
      cp_async_commit();
    }
  }
  for (int k = tid; k < K; k += kT) store_row_value(a, (size_t)grow * LD + k, x_s[k]);
  if (a.pc_out) {
#pragma unroll
    for (int m = 0; m < MW; m++) {
      const int j = m * kT + tid;
      if (j < n) pc_store(a, p0 + j, pr[m]);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Heavy rows: slabs of kSlab nonzeros, prediction cache in HBM (a compact array per side), one
// launch pair per factor block over a BATCH of rows small enough that the block's lines stay in L2
// between the partials launch and the deferred cache update of the next one.
// ---------------------------------------------------------------------------------------------
// One slab ("unit") of a heavy row, 32 bytes: read with two 16-byte loads at the top of the kernel.
struct __align__(16) UnitDesc {
  int64_t off;      // offset of the unit's first nonzero in the side's idx/val arrays
  int64_t poff;     // offset of the same nonzero in the compact prediction cache
  int32_t cnt;      // nonzeros in the unit (<= slab size)
  int32_t row;      // owned-row id
  int32_t hrow;     // index of that row among the heavy rows (delta / x slots)
  int32_t slot;     // canonical unit id = slot of its partial sums
};

struct HeavyUnits {
  // Descriptors of the units a launch covers, in LAUNCH order (CTA b takes units[b]).  Canonical
  // order is row by row; the launch order of a whole batch sorts the slabs by the id of their FIRST
  // neighbour, so that CTAs running at the same time gather (largely) the same neighbour rows: with
  // every heavy row of a side in one batch, a neighbour's line is fetched from HBM once per step
  // and served to the other slabs — and to the deferred cache update of the next step — from L2
  // (before: 243 B of DRAM reads per nonzero and block, L2 hit rate 9 %; profiles/README.md r01f/h).
  const UnitDesc* units;
  const int32_t* hrow_id;      // owned-row id of heavy row h
  const int32_t* hrow_grp0;    // first reduction group of heavy row h (groups of <= 32 consecutive units)
  const int32_t* hrow_grps;    // number of groups of heavy row h
  const int32_t* grp_unit0;    // first unit (canonical id) of group g
  const int32_t* grp_cnt;      // units in group g
};

__device__ __forceinline__ UnitDesc load_unit(const UnitDesc* p) {
  const int4 a = __ldg(reinterpret_cast<const int4*>(p));
  const int4 b = __ldg(reinterpret_cast<const int4*>(p) + 1);
  UnitDesc d;
  d.off = ((int64_t)(uint32_t)a.y << 32) | (uint32_t)a.x;
  d.poff = ((int64_t)(uint32_t)a.w << 32) | (uint32_t)a.z;
  d.cnt = b.x; d.row = b.y; d.hrow = b.z; d.slot = b.w;
  return d;
}

// p_j = <x_row, y_j> for every nonzero of the units [u0, u0 + gridDim.x): 8 lanes per nonzero.
template <int LD>
__global__ void __launch_bounds__(kBlkThreads)
heavy_pred_kernel(CdSide a, HeavyUnits hu, double* __restrict__ pred) {
  __shared__ double x_s[LD];
  const int tid = threadIdx.x;
  const UnitDesc ud = load_unit(hu.units + blockIdx.x);
  const int row = ud.row;
  const double* xrow = a.X + (size_t)(a.row_base + row) * LD;
  for (int k = tid; k < LD; k += kBlkThreads) x_s[k] = xrow[k];
  __syncthreads();
  const int64_t off = ud.off, poff = ud.poff;
  const int cnt = ud.cnt;
  const int g8 = tid >> 3, gl = tid & 7;
  for (int j0 = 0; j0 < cnt; j0 += kBlkThreads / 8) {   // cnt <= kMaxSlab
    const int j = j0 + g8;
    double acc = 0.0;
    if (j < cnt) {
      const double* yrow = a.Y + (size_t)a.idx[off + j] * LD;
#pragma unroll
      for (int c = 0; c < LD; c += kFB) {
        const double2 d = ldg2(yrow + c + gl * 2);
        acc += x_s[c + gl * 2] * d.x;
        acc += x_s[c + gl * 2 + 1] * d.y;
      }
    }
    acc += __shfl_xor_sync(kFullMask, acc, 1);
    acc += __shfl_xor_sync(kFullMask, acc, 2);
    acc += __shfl_xor_sync(kFullMask, acc, 4);
    if (j < cnt && gl == 0) pred[poff + j] = acc;
  }
}

template <int SLAB>
struct HeavySmem {
  static constexpr size_t kTile = (size_t)SLAB * 128;       // x2: previous block (cache update) + this block
  static constexpr size_t kIdx = (size_t)SLAB * 8;          // row base pointers
  static constexpr size_t kCZ = (size_t)SLAB * 16;
  // the per-warp reduction slots (SLAB/32 x 208 doubles) reuse the previous-block tile once it is consumed
  static constexpr size_t kBytes = 2 * kTile + kIdx + kCZ + 16 * 8;
  static_assert((size_t)(SLAB / 32) * kPartLen * 8 <= kTile, "slots must fit the spare tile");
};

// Step fb of the batch: (1) if fb > 0, apply the cache update of block fb-1 (needs that block's
// lines again); (2) if fb < nblocks, form the slab's partial Gram and right-hand side of block fb
// (tensor cores) and write them to partials[slot].  Both tiles are requested up front in one pass
// over the row pointers, so a slab pays one memory round trip per step, not two; the slab descriptor is
// one 32-byte record in launch order, so the dependent chain is descriptor -> indices -> gather.
// One nonzero per thread: SLAB threads per CTA (256: 3 CTAs/SM, 128: 6 CTAs/SM).
template <int LD, bool USER, int SLAB>
__global__ void __launch_bounds__(SLAB, SLAB == 256 ? 3 : 6)
heavy_step_kernel(CdSide a, HeavyUnits hu, int u0, int fb, int nblocks, double* __restrict__ pred,
                  const double* __restrict__ delta, double* __restrict__ partials) {
  extern __shared__ __align__(128) unsigned char smem[];
  using Sm = HeavySmem<SLAB>;
  unsigned char* tile_prev = smem;
  unsigned char* tile = smem + Sm::kTile;
  const double** rowp_s = reinterpret_cast<const double**>(smem + 2 * Sm::kTile);
  double* c_s = reinterpret_cast<double*>(smem + 2 * Sm::kTile + Sm::kIdx);
  double* z_s = c_s + SLAB;
  double* delta_s = z_s + SLAB;
  double* slots = reinterpret_cast<double*>(tile_prev);   // free again after the cache update

  const int tid = threadIdx.x, lane = lane_id(), warp = tid >> 5;
  const UnitDesc ud = load_unit(hu.units + blockIdx.x);
  const int64_t off = ud.off, poff = ud.poff;
  const int n = ud.cnt;
  const int n_pad = (n + 3) & ~3;
  const int grow = a.row_base + ud.row;
  const double wi_row = USER ? 0.0 : a.Wi[grow];

  double pr = 0.0, cw = 0.0, wr = 0.0;
  if (tid < n) {
    const int id = a.idx[off + tid];
    rowp_s[tid] = a.Y + (size_t)id * LD;
    const double w = a.val ? a.val[off + tid] : 1.0;
    wr = w * w;
    cw = w - (USER ? a.Wi[id] : wi_row);
    pr = (fb == 0 && a.use_cache) ? a.pc_in[off + tid] : pred[poff + tid];
  }
  c_s[tid] = cw;
  if (fb > 0 && tid < 16) delta_s[tid] = delta[(size_t)ud.hrow * 16 + tid];
  __syncthreads();

  stage_two_tiles(tile_prev, tile, rowp_s, n, n_pad, fb, fb > 0, fb < nblocks, tid, SLAB);
  cp_async_commit();
  if (fb > 0) {
    cp_async_wait<0>();
    __syncthreads();
    if (tid < n) {
      double y[16];
      load_tile_row(tile_prev, tid, y);
      double a0 = pr, a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll
      for (int e = 0; e < 16; e += 4) {
        a0 += delta_s[e] * y[e];
        a1 += delta_s[e + 1] * y[e + 1];
        a2 += delta_s[e + 2] * y[e + 2];
        a3 += delta_s[e + 3] * y[e + 3];
      }
      pr = (a0 + a1) + (a2 + a3);
      if (fb < nblocks) pred[poff + tid] = pr;
      else if (a.pc_out) pc_store(a, off + tid, pr);   // final value -> symmetric cache
    }
  } else if (a.use_cache && tid < n) {
    pred[poff + tid] = pr;   // the pipeline's compact cache starts from the symmetric one
  }
  if (fb >= nblocks) return;
  z_s[tid] = tid < n ? wr - cw * pr : 0.0;
  if (fb == 0) cp_async_wait<0>();
  __syncthreads();   // z_s (and, for fb = 0, the tile) visible; every thread is done with tile_prev

  double frag[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  gram_rhs_fragments(tile, c_s, z_s, warp * 32, min(warp * 32 + 32, n_pad), frag);
  double* slot = slots + warp * kPartLen;
#pragma unroll
  for (int t = 0; t < 3; t++) {
    slot[t * 64 + lane * 2] = frag[2 * t];
    slot[t * 64 + lane * 2 + 1] = frag[2 * t + 1];
  }
  if ((lane & 3) == 0) {
    slot[192 + (lane >> 2)] = frag[6];
    slot[200 + (lane >> 2)] = frag[8];
  }
  __syncthreads();
  for (int i = tid; i < kPartLen; i += SLAB) {
    double sum = 0.0;
#pragma unroll
    for (int w = 0; w < SLAB / 32; w++) sum += slots[w * kPartLen + i];
    partials[(size_t)(ud.slot - u0) * kPartLen + i] = sum;
  }
}

// Level-1 reduction: out[g - g0] = sum of the unit partials of group g (<= 32 consecutive units of one
// row), added in unit order.
__global__ void __launch_bounds__(kBlkThreads)
heavy_reduce_kernel(const double* __restrict__ partials, HeavyUnits hu, int g0, int u0, double* __restrict__ out) {
  const int tid = threadIdx.x;
  if (tid >= kPartLen) return;
  const int g = g0 + blockIdx.x;
  const int q0 = hu.grp_unit0[g] - u0, q1 = q0 + hu.grp_cnt[g];
  double s = 0.0;
  for (int q = q0; q < q1; q++) s += partials[(size_t)q * kPartLen + tid];
  out[(size_t)blockIdx.x * kPartLen + tid] = s;
}

// One CTA per heavy row of the batch: add the row's partials in a fixed order (8 warps take every
// 8th entry, then the 8 sums are added in warp order) while all threads form S.x of the block;
// warp 0 then runs the 16-step recurrence; the new factors and d_f go to HBM.
// partials = the group sums of the batch (heavy_reduce_kernel), group g at slot g - g0.
template <int LD, bool USER>
__global__ void __launch_bounds__(kBlkThreads)
heavy_solve_kernel(CdSide a, HeavyUnits hu, int h0, int g0, int fb, const double* __restrict__ partials,
                   double* __restrict__ delta) {
  __shared__ double x_s[LD];
  __shared__ double Gs[kGsLen];
  __shared__ double Pt[16];
  __shared__ double Tt[16];
  __shared__ double tpart[16][16];
  __shared__ double wsum[kBlkWarps][kPartLen];
  const int tid = threadIdx.x, lane = lane_id(), warp = tid >> 5;
  const int h = h0 + blockIdx.x;
  const int row = hu.hrow_id[h];
  const int grow = a.row_base + row;
  const int f0 = fb * kFB;
  const double g = USER ? 1.0 : a.Wi[grow];
  double* xrow = a.X + (size_t)grow * LD;
  for (int k = tid; k < LD; k += kBlkThreads) x_s[k] = xrow[k];
  const int ufirst = hu.hrow_grp0[h] - g0;
  const int ucount = hu.hrow_grps[h];
  {
    double acc[7];
#pragma unroll
    for (int t = 0; t < 7; t++) acc[t] = 0.0;
    for (int q = warp; q < ucount; q += kBlkWarps) {
      const double* p = partials + (size_t)(ufirst + q) * kPartLen;
#pragma unroll
      for (int t = 0; t < 7; t++)
        if (lane + 32 * t < kPartLen) acc[t] += p[lane + 32 * t];
    }
#pragma unroll
    for (int t = 0; t < 7; t++)
      if (lane + 32 * t < kPartLen) wsum[warp][lane + 32 * t] = acc[t];
  }
  __syncthreads();
  {   // S.x: thread = (factor, 1/16th of the k range); S symmetric -> unit stride over the factor
    constexpr int kPer = LD / 16;
    const int tf = tid & 15, part = tid >> 4;
    const double* __restrict__ Sc = a.S + (size_t)(part * kPer) * LD + f0 + tf;
    double t0 = 0.0, t1 = 0.0;
#pragma unroll 8
    for (int k = 0; k < kPer; k += 2) {
      t0 += x_s[part * kPer + k] * __ldg(Sc + (size_t)k * LD);
      if (kPer > 1) t1 += x_s[part * kPer + k + 1] * __ldg(Sc + (size_t)(k + 1) * LD);
    }
    tpart[part][tf] = t0 + t1;
  }
  if (tid < kPartLen) {
    double sum = 0.0;
#pragma unroll
    for (int w = 0; w < kBlkWarps; w++) sum += wsum[w][tid];
    if (tid < 192) {   // H = G + g S_BB
      const int t = tid >> 6, l = (tid & 63) >> 1, ii = tid & 1;
      int rw = l >> 2, cl = 2 * (l & 3) + ii;
      if (t >= 1) rw += 8;
      if (t == 2) cl += 8;
      sum += g * __ldg(a.S + (size_t)(f0 + rw) * LD + f0 + cl);
      Gs[rw * kGsStride + cl] = sum;
    } else {
      Pt[tid - 192] = sum;
    }
  }
  __syncthreads();
  if (tid < 16) {
    double sum = 0.0;
#pragma unroll
    for (int q = 0; q < 16; q++) sum += tpart[q][tid];
    Tt[tid] = sum;
  }
  __syncthreads();
  if (warp == 0) {
    const int ff = lane & 15;
    double hcol[16];
#pragma unroll
    for (int k = 0; k < 16; k++) hcol[k] = Gs[ff * kGsStride + k];
    const double hff = Gs[ff * kGsStride + ff];
    const double xf = x_s[f0 + ff];
    double numer = Pt[ff] - g * Tt[ff] + xf * hff;
    const double rden = 1.0 / (hff + a.reg);
#pragma unroll
    for (int sidx = 0; sidx < 16; sidx++) {
      const double d = numer * rden - xf;
      const double ds = __shfl_sync(kFullMask, d, sidx);
      if (ff > sidx) numer -= ds * hcol[sidx];
    }
    const double xnew = numer * rden;
    if (lane < 16) {
      const bool livef = f0 + ff < a.K;
      delta[(size_t)h * 16 + ff] = livef ? xnew - xf : 0.0;
      if (livef) store_row_value(a, (size_t)grow * LD + f0 + ff, xnew);
    }
  }
}

}  // namespace eals
