// eval_tc.cuh — K3 on the 5th-generation tensor cores: the blocked U.V^T scoring pass of the
// leave-one-out evaluation (MF_fastALS::evaluate_for_user, MF_fastALS.cpp:620-662, driven over all
// users by evaluate_model, main.cpp:37-65) as a tcgen05 FILTER in front of the exact fp64 test.
//
// What must come out is decided by exact fp64 comparisons (score(u,i) > score(u,gt), strict, with the
// reference's sequential-k sums — eval.cuh), and one flipped user moves HR by 1/M.  So the tensor
// pass never decides a close call.  Both factor matrices are scaled by powers of two (U per row, V by
// one global exponent; exact) and rounded to fp16; the kernel below forms acc = sum_k uh_k vh_k on
// tcgen05.mma (fp16 x fp16 products are exact in fp32, fp32 accumulation in TMEM) and compares it
// with thresholds that carry a RIGOROUS error bound E(u, item tile):
//
//     |acc - s^|  <=  |du|.|vh| + |u^|.|dv| + gamma.(|uh|+|du|).(|vh|+|dv|)  =: E
//
// (s^ = the reference's fp64 score in the scaled domain, du = uh - u^ the ACTUAL rounding error
// vector of the row, norms are 2-norms rounded up, the maxima over the 128 items of a tile stand in for
// the item norms; gamma = KP.2^-21 covers fp32 accumulation with truncation four times over plus the
// fp64 rounding of the reference's own sum).  Then
//
//     acc >  g^ + E   =>  score > gt score for certain          (counted here, MODE 0)
//     acc <  g^ - E   =>  score <= gt score for certain         (dropped)
//     otherwise       =>  candidate: re-scored in fp64 with the reference's operation order (MODE 1 emits
//                         the pair; eval_rescore_kernel decides)
//
// A user whose CERTAIN count exceeds topK is out (the reference returns zeros, :633-634) without a
// single exact score; the survivors' candidates — a sliver of the catalogue each — are re-scored exactly,
// so count_larger, HR, NDCG and the reciprocal rank are identical to the all-fp64 scan (tested).  Items
// are visited in order of decreasing norm: the tile maxima are tight and the high scorers come first, so
// most users are decided in the first item block and leave the working set.
//
// Kernel anatomy (persistent, one CTA per SM, 320 threads):
//   warp 0      TMA producer: the UT user tiles of a work item once, then the item tiles through an
//               S-stage shared-memory ring (cp.async.bulk.tensor, 128-byte swizzle, mbarrier tx counts)
//   warp 1      tcgen05.mma issuer (one lane): per stage UT x (KP/16) MMAs of 128 x 128 x 16 into one of
//               two TMEM accumulator buffers; tcgen05.commit releases the stage and publishes the buffer
//   warps 2-9   epilogue: tcgen05.ld of the warp's 32 TMEM lanes (= 32 users) x 64 columns, compare against
//               the per-(user, tile) thresholds, count in registers (MODE 0) or emit candidates (MODE 1; MODE 2
//               for recommend.cuh: acc >= t^ - E only, t^ = the user's k-th score in place of the gt score)
// Two user tiles share every staged item tile (UT = 2 for K <= 128): 32 bytes of L2 traffic per SM and
// clock instead of 64, which is what keeps 148 SMs under the L2 fabric's ~6300 B/clk.  The host walks
// the catalogue in L2-sized item blocks and compacts the working set between them on the device.
#pragma once

#include <cuda.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "eval.cuh"

namespace eals {
namespace tc {

constexpr int kTM = 128;             // users per accumulator tile (UMMA M)
constexpr int kTN = 128;             // items per stage (UMMA N)
constexpr int kKC = 64;              // halves per 128-byte swizzle row
constexpr int kChunk = 128 * 128;    // bytes of one [128 rows][64 halves] swizzled sub-tile
constexpr int kThreads = 320;           // TMA warp + MMA warp + 8 epilogue warps

template <int NKC>
struct Cfg {
  static constexpr int UT = NKC <= 2 ? 2 : 1;   // user tiles per work item
  static constexpr int S = NKC == 1 ? 8 : (NKC == 2 ? 4 : (NKC == 3 ? 3 : 2));
  static constexpr size_t kU = (size_t)UT * NKC * kChunk;
  static constexpr size_t kStage = (size_t)NKC * kChunk;
  static constexpr size_t kBar = 256;
  static constexpr int kStagePairs = 224;                          // MODE 1: candidate pairs staged per epilogue warp
  static constexpr size_t kEmit = 8 * (size_t)kStagePairs * 16;
  static constexpr size_t kSmem = 1024 + kU + S * kStage + kBar;   // 1024: alignment slack for the swizzle atoms
  static constexpr size_t kSmemEmit = kSmem + kEmit;
  static constexpr int kTmemCols = 512;
};

struct EvalPair {
  int32_t slot;    // position in the caller's user list
  int32_t item;    // item id (original order)
  int32_t flags;   // bit 0: candidate for "score > gt score"; bit 1: candidate for "(int)score != 0"
  int32_t key;     // (int)score, filled by the exact pass
};

struct TcArgs {
  const int32_t* act;          // working list: position -> slot (nullptr: identity)
  const int32_t* n_act;        // device scalar: positions in the working list
  const float4* sp0;           // per slot {g^ rounded up, g^ rounded down, |u^|, |du|}
  const float4* sp1;           // per slot {gamma (|uh| + |du|), 2^-(e_u + e_V), 0, 0}
  const float2* tile_norm;     // per item tile {max |vh|, max |dv|}
  int it0, it1;                // item tiles [it0, it1) of the norm-sorted catalogue
  int n_items;
  int32_t* cnt_hi;             // MODE 0: certain count per slot (accumulated over item blocks)
  const int32_t* perm;         // MODE 1: sorted rank -> item id
  EvalPair* pairs;
  unsigned long long* n_pairs;
  unsigned long long cap_pairs;
};

// ---- PTX wrappers ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n.reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {}
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cta.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n"
               ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem] . B[smem]^T, one 128 x 128 x 16 fp16 step; fp32 accumulate.
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread t of the warp gets TMEM lane (base lane + t).  The values
// may only be read after tc_ld_wait().
__device__ __forceinline__ void tc_ld32_issue(uint32_t taddr, float (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]),
        "=f"(v[8]), "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15]),
        "=f"(v[16]), "=f"(v[17]), "=f"(v[18]), "=f"(v[19]), "=f"(v[20]), "=f"(v[21]), "=f"(v[22]), "=f"(v[23]),
        "=f"(v[24]), "=f"(v[25]), "=f"(v[26]), "=f"(v[27]), "=f"(v[28]), "=f"(v[29]), "=f"(v[30]), "=f"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }

// Shared-memory matrix descriptor of a K-major, 128-byte-swizzled operand tile (rows of 64 halves, 8-row
// groups 1024 bytes apart): start address >> 4 | LBO = 1 (ignored for swizzled K-major) | SBO = 1024 >> 4 |
// version 1 (Blackwell) | layout SWIZZLE_128B.
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor, kind::f16: D = fp32 (bits 4-5 = 1), A = B = fp16 (0), both K-major, N >> 3 at bit 17,
// M >> 4 at bit 24.
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- the filter kernel ------------------------------------------------------------------------------
template <int NKC, int MODE>
__global__ void __launch_bounds__(kThreads, 1)
eval_filter_kernel(const __grid_constant__ CUtensorMap mapU, const __grid_constant__ CUtensorMap mapV, TcArgs a) {
  using C = Cfg<NKC>;
  constexpr int UT = C::UT, S = C::S;
  extern __shared__ unsigned char smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t u_smem = base;
  const uint32_t v_smem = base + (uint32_t)C::kU;
  const uint32_t bars = v_smem + (uint32_t)(S * C::kStage);
  // barriers: full[S], empty[S], u_full, u_empty, acc_full[2], acc_empty[2]; then the TMEM base address slot
  const uint32_t bar_full = bars, bar_empty = bars + 8 * S, bar_ufull = bars + 16 * S, bar_uempty = bar_ufull + 8;
  const uint32_t bar_accfull = bar_uempty + 8, bar_accempty = bar_accfull + 16;
  const uint32_t tmem_slot = bar_accempty + 16;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < S; s++) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
    mbar_init(bar_ufull, 1); mbar_init(bar_uempty, 1);
    for (int b = 0; b < 2; b++) { mbar_init(bar_accfull + 8 * b, 1); mbar_init(bar_accempty + 8 * b, 8); }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(tmem_slot), "r"(C::kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  const int n_act = *a.n_act;
  // Work item = (group of UT user tiles, chunk of the item-tile range).  With many user tiles a work item
  // walks the whole range (chunks = 1: the user tiles are loaded once); when the working set has shrunk to a
  // few tiles the range is cut so that every SM still gets ~4 work items (the candidate pass over 40k users
  // of a 10M-user evaluation was two waves of 148 + 8 CTAs walking 15,625 tiles each before this).
  const int n_uw = (n_act + UT * kTM - 1) / (UT * kTM);
  const int n_it_all = a.it1 - a.it0;
  int chunks = 1;
  if (n_uw > 0 && n_uw < 4 * (int)gridDim.x) chunks = (4 * (int)gridDim.x + n_uw - 1) / n_uw;
  chunks = max(1, min(chunks, (n_it_all + 15) / 16));
  const int tpc = (n_it_all + chunks - 1) / chunks;
  chunks = (n_it_all + tpc - 1) / tpc;
  const int n_works = n_uw * chunks;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0, uphase = 0;
      for (int w = blockIdx.x; w < n_works; w += gridDim.x) {
        const int uw = w / chunks, tb = (w % chunks) * tpc, n_it = min(tpc, n_it_all - tb);
        const int it_base = a.it0 + tb;
        mbar_wait(bar_uempty, uphase ^ 1);
        mbar_expect_tx(bar_ufull, (uint32_t)C::kU);
#pragma unroll
        for (int j = 0; j < UT; j++)
#pragma unroll
          for (int kc = 0; kc < NKC; kc++)
            tma_load_2d(u_smem + (uint32_t)((j * NKC + kc) * kChunk), &mapU, kc * kKC, (uw * UT + j) * kTM, bar_ufull);
        for (int t = 0; t < n_it; t++) {
          mbar_wait(bar_empty + 8 * stage, phase ^ 1);
          mbar_expect_tx(bar_full + 8 * stage, (uint32_t)C::kStage);
#pragma unroll
          for (int kc = 0; kc < NKC; kc++)
            tma_load_2d(v_smem + (uint32_t)(stage * C::kStage + kc * kChunk), &mapV, kc * kKC, (it_base + t) * kTN, bar_full + 8 * stage);
          if (++stage == S) { stage = 0; phase ^= 1; }
        }
        uphase ^= 1;
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    constexpr uint32_t idesc = umma_idesc_f16(kTM, kTN);
    int stage = 0, ab = 0;
    uint32_t phase = 0, uphase = 0, aphase = 0;
    for (int w = blockIdx.x; w < n_works; w += gridDim.x) {
      const int n_it = min(tpc, n_it_all - (w % chunks) * tpc);
      mbar_wait(bar_ufull, uphase);
      tc_fence_after();
      for (int t = 0; t < n_it; t++) {
        mbar_wait(bar_accempty + 8 * ab, aphase ^ 1);   // the epilogue has drained this accumulator buffer
        mbar_wait(bar_full + 8 * stage, phase);         // the item tile has landed
        tc_fence_after();
        if (lane == 0) {
#pragma unroll
          for (int j = 0; j < UT; j++) {
            const uint32_t d = tmem_base + (uint32_t)((ab * UT + j) * kTN);
#pragma unroll
            for (int kc = 0; kc < NKC; kc++)
#pragma unroll
              for (int k = 0; k < 4; k++) {
                const uint64_t da = umma_desc(u_smem + (uint32_t)((j * NKC + kc) * kChunk + k * 32));
                const uint64_t db = umma_desc(v_smem + (uint32_t)(stage * C::kStage + kc * kChunk + k * 32));
                tc_mma_f16(d, da, db, idesc, (kc | k) != 0 ? 1u : 0u);
              }
          }
          tc_commit(bar_empty + 8 * stage);      // stage reusable once these MMAs have read it
          tc_commit(bar_accfull + 8 * ab);       // accumulators complete
        }
        __syncwarp();
        if (++stage == S) { stage = 0; phase ^= 1; }
        if (++ab == 2) { ab = 0; aphase ^= 1; }
      }
      if (lane == 0) tc_commit(bar_uempty);      // user tiles reusable after the last MMA of this work item
      __syncwarp();
      uphase ^= 1;
    }
  } else {
    // ===== epilogue: warps 2..9.  TMEM lane quadrant q = warp & 3 (a warp may only touch lanes 32 q .. 32 q + 31 =
    // 32 users), column half hf = (warp - 2) >> 2 (64 of the 128 items of a tile).  Eight warps, two per scheduler,
    // and both TMEM loads of a (tile, user tile) in flight before the first wait: with four warps and a wait after
    // every load the compare loop, not the tensor pipe, set the pace (2.7k cycles per tile against 1k; r2f). =====
    const int q = warp & 3, hf = (warp - 2) >> 2;
    constexpr int kCols = kTN / 2;                       // columns per epilogue warp
    int ab = 0;
    uint32_t aphase = 0;
    // MODE 1: this warp's staging buffer for candidate pairs (flushed to the global list with one atomic)
    EvalPair* stage_buf = reinterpret_cast<EvalPair*>(smem_raw + (bars + (uint32_t)C::kBar - smem_u32(smem_raw))) + (warp - 2) * C::kStagePairs;
    int fill = 0;
    auto flush = [&]() {
      __syncwarp();
      if (fill > 0) {
        unsigned long long fb = 0;
        if (lane == 0) fb = atomicAdd(a.n_pairs, (unsigned long long)fill);
        fb = __shfl_sync(kFullMask, fb, 0);
        for (int i = lane; i < fill; i += 32)
          if (fb + i < a.cap_pairs) a.pairs[fb + i] = stage_buf[i];
      }
      fill = 0;
      __syncwarp();
    };
    for (int w = blockIdx.x; w < n_works; w += gridDim.x) {
      const int uw = w / chunks, tb = (w % chunks) * tpc, n_it = min(tpc, n_it_all - tb);
      float ghi[UT], glo[UT], na[UT], nd[UT], ns[UT], one[UT];
      int slot[UT], cnt[UT];
#pragma unroll
      for (int j = 0; j < UT; j++) {
        const int p = (uw * UT + j) * kTM + q * 32 + lane;
        slot[j] = -1; cnt[j] = 0;
        ghi[j] = glo[j] = na[j] = nd[j] = ns[j] = one[j] = 0.f;
        if (p < n_act) {
          slot[j] = a.act ? a.act[p] : p;
          const float4 s0 = a.sp0[slot[j]], s1 = a.sp1[slot[j]];
          ghi[j] = s0.x; glo[j] = s0.y; na[j] = s0.z; nd[j] = s0.w; ns[j] = s1.x; one[j] = s1.y;
        }
      }
      for (int t = 0; t < n_it; t++) {
        const int it = a.it0 + tb + t;
        const float2 tn = __ldg(a.tile_norm + it);
        const int nvalid = a.n_items - it * kTN - hf * kCols;      // valid columns of this warp's half (< 64 only at the end)
        mbar_wait(bar_accfull + 8 * ab, aphase);
        tc_fence_after();
#pragma unroll
        for (int j = 0; j < UT; j++) {
          // E = |du| max|vh| + |u^| max|dv| + gamma (|uh| + |du|) (max|vh| + max|dv|), every step rounded up
          const float E = __fmaf_ru(nd[j], tn.x, __fmaf_ru(na[j], tn.y, __fmul_ru(ns[j], __fadd_ru(tn.x, tn.y))));
          const float thr_hi = slot[j] >= 0 ? __fadd_ru(ghi[j], E) : __int_as_float(0x7f800000);
          const float thr_lo = __fsub_rd(glo[j], E);
          const float thr_one = __fsub_rd(one[j], E);
          const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((ab * UT + j) * kTN + hf * kCols);
          float v[kCols];
          tc_ld32_issue(taddr, *reinterpret_cast<float(*)[32]>(&v[0]));
          tc_ld32_issue(taddr + 32, *reinterpret_cast<float(*)[32]>(&v[32]));
          tc_ld_wait();
          if (MODE == 0) {
            if (nvalid >= kCols) {
#pragma unroll
              for (int i = 0; i < kCols; i++) cnt[j] += v[i] > thr_hi ? 1 : 0;
            } else {
#pragma unroll
              for (int i = 0; i < kCols; i++) cnt[j] += (i < nvalid && v[i] > thr_hi) ? 1 : 0;
            }
          } else {
            // candidate masks: bit i of m1 = "may exceed the gt score", of m2 = "|score| may reach 1".  Almost every
            // lane has no candidate in a given tile (0.04 per lane and tile at 10M x 2M), so a two-compare screen
            // per score comes first and the masks are only built by the lanes that need them.
            // MODE 2 (recommend): only "may reach the user's k-th score" (thr_lo); no |score| >= 1 clause.
            uint32_t m1[2] = {0u, 0u}, m2[2] = {0u, 0u};
            const float t_pos = MODE == 2 ? thr_lo : fminf(thr_lo, thr_one);
            const float t_neg = MODE == 2 ? -__int_as_float(0x7f800000) : -thr_one;
            bool hit = false;
#pragma unroll
            for (int i = 0; i < kCols; i++) hit |= (v[i] >= t_pos) | (v[i] <= t_neg);
            if (hit && slot[j] >= 0) {
#pragma unroll
              for (int c = 0; c < 2; c++) {
                uint32_t b1 = 0, b2 = 0;
#pragma unroll
                for (int i = 0; i < 32; i++) {
                  b1 |= (v[c * 32 + i] >= thr_lo ? 1u : 0u) << i;
                  if (MODE == 1) b2 |= (fabsf(v[c * 32 + i]) >= thr_one ? 1u : 0u) << i;
                }
                const int lim = nvalid - c * 32;
                const uint32_t live = lim <= 0 ? 0u : (lim >= 32 ? 0xffffffffu : ((1u << lim) - 1u));
                m1[c] = b1 & live;
                m2[c] = b2 & live;
              }
            }
            // Warp-aggregated append into this warp's shared-memory staging buffer; the buffer goes to the global
            // list with ONE atomic per flush (one atomic per pair — ~700 dependent atomics per thread — made this
            // pass 1.9 s of a 5 s evaluation at 10M x 2M; one per warp and tile still 0.26 s: profiles r2d / r2e).
            // Tried and dropped: one warp vote per COLUMN instead of per-lane masks + scan — 64 unrolled copies
            // of the append path per user tile: 457 ms instead of 61 (r02n).
            const int mine = __popc(m1[0] | m2[0]) + __popc(m1[1] | m2[1]);
            int incl = mine;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
              const int up = __shfl_up_sync(kFullMask, incl, o);
              if (lane >= o) incl += up;
            }
            const int total = __shfl_sync(kFullMask, incl, 31);
            if (total > 0) {
              if (fill + total > C::kStagePairs) flush();
              const bool direct = total > C::kStagePairs;          // more than the buffer holds: straight to the list
              unsigned long long wbase = 0;
              if (direct) {
                if (lane == 0) wbase = atomicAdd(a.n_pairs, (unsigned long long)total);
                wbase = __shfl_sync(kFullMask, wbase, 0);
              }
              int at = fill + incl - mine;
#pragma unroll
              for (int c = 0; c < 2; c++) {
                uint32_t any = m1[c] | m2[c];
                while (any) {
                  const int i = __ffs(any) - 1;
                  any &= any - 1;
                  const int fl = ((m1[c] >> i) & 1) | (((m2[c] >> i) & 1) << 1);
                  const EvalPair pr{slot[j], a.perm[it * kTN + hf * kCols + c * 32 + i], fl, 0};
                  if (!direct) stage_buf[at] = pr;
                  else if (wbase + (unsigned long long)(at - fill) < a.cap_pairs) a.pairs[wbase + (unsigned long long)(at - fill)] = pr;
                  at++;
                }
              }
              if (!direct) fill += total;
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_accempty + 8 * ab);
        if (++ab == 2) { ab = 0; aphase ^= 1; }
      }
      if (MODE == 0) {
#pragma unroll
        for (int j = 0; j < UT; j++)
          if (slot[j] >= 0 && cnt[j]) atomicAdd(a.cnt_hi + slot[j], cnt[j]);   // two column halves (and item chunks) per slot
      } else {
        flush();
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(C::kTmemCols) : "memory");
  }
}

// ---- preparation kernels ----------------------------------------------------------------------------
// exponent e with |x| * 2^-e in [1, 2) for the largest |x| of the row (0 for an all-zero row)
__device__ __forceinline__ int exponent_of(double amax) {
  if (!(amax > 0.0)) return 0;
  int e;
  frexp(amax, &e);   // amax = m * 2^e, m in [0.5, 1)
  return e - 1;
}

// max |x| over a [rows][LD] matrix (first K columns) -> *out as the bit pattern of a non-negative double
__global__ void absmax_kernel(const double* __restrict__ X, size_t rows, int K, int LD, unsigned long long* __restrict__ out) {
  double m = 0.0;
  const size_t total = rows * (size_t)LD;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x)
    if ((int)(t % LD) < K) m = fmax(m, fabs(X[t]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(kFullMask, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.0) atomicMax(out, (unsigned long long)__double_as_longlong(m));
}

// One warp per row: scale by 2^-e (e per row when row_exp == nullptr... see below), round to fp16, write the
// row padded with zeros to KP halves, and the three norms (fp32, rounded up).
//   USERS: e = exponent of the row's own max; also the per-slot thresholds from the exact gt score.
//   ITEMS: e = the global exponent *e_glob; rows are written in sorted order (src row = perm[r]).
struct PrepOut {
  __half* H;             // [rows][KP]
  float* n_hat;          // |x^|  (scaled, unrounded)
  float* n_del;          // |xh - x^|
  float* n_h;            // |xh|
  int* exps;             // per-row exponent (users)
};

template <bool USERS>
__global__ void prep_rows_kernel(const double* __restrict__ X, int K, int LD, int KP, int rows,
                                 const int32_t* __restrict__ src_row,   // USERS: slot -> user id (nullable: base + r); ITEMS: rank -> item
                                 int row_base, const unsigned long long* __restrict__ glob_absmax, PrepOut o) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const int src = src_row ? src_row[warp] : row_base + warp;
  const double* x = X + (size_t)src * LD;
  double amax = 0.0;
  if (USERS) {
    for (int k = lane; k < K; k += 32) amax = fmax(amax, fabs(x[k]));
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) amax = fmax(amax, __shfl_xor_sync(kFullMask, amax, off));
  } else {
    amax = __longlong_as_double((long long)*glob_absmax);
  }
  const int e = exponent_of(amax);
  double s_hat = 0.0, s_del = 0.0, s_h = 0.0;
  __half* h = o.H + (size_t)warp * KP;
  for (int k = lane; k < KP; k += 32) {
    double xs = 0.0;
    __half hv = __float2half_rn(0.f);
    if (k < K) {
      xs = ldexp(x[k], -e);              // exact (power of two)
      hv = __double2half(xs);            // round to nearest even, straight from fp64
      const double back = (double)__half2float(hv);
      s_hat += xs * xs;
      s_del += (back - xs) * (back - xs);
      s_h += back * back;
    }
    h[k] = hv;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    s_hat += __shfl_xor_sync(kFullMask, s_hat, off);
    s_del += __shfl_xor_sync(kFullMask, s_del, off);
    s_h += __shfl_xor_sync(kFullMask, s_h, off);
  }
  if (lane == 0) {
    // fp64 sums of <= 256 squares are good to ~1e-14 relative; the factor below dwarfs that, then round up
    const double up = 1.0 + 1e-9;
    o.n_hat[warp] = __double2float_ru(sqrt(s_hat) * up);
    o.n_del[warp] = __double2float_ru(sqrt(s_del) * up);
    o.n_h[warp] = __double2float_ru(sqrt(s_h) * up);
    if (o.exps) o.exps[warp] = e;
  }
}

// Per-slot filter parameters from the exact gt score (eval_gt_score_kernel) and the row norms.
__global__ void slot_params_kernel(const double* __restrict__ gt_score, const int* __restrict__ exps, const unsigned long long* __restrict__ v_absmax,
                                   const float* __restrict__ n_hat, const float* __restrict__ n_del, const float* __restrict__ n_h,
                                   int n, double gamma, float4* __restrict__ sp0, float4* __restrict__ sp1) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  const int ev = exponent_of(__longlong_as_double((long long)*v_absmax));
  const int e = exps[s] + ev;
  const double gh = ldexp(gt_score[s], -e);
  const double one = ldexp(1.0, -e);
  float one_f = __double2float_rd(one);
  if (!(one_f > 0.f)) one_f = 1e-45f;                       // never "everything qualifies"
  sp0[s] = make_float4(__double2float_ru(gh), __double2float_rd(gh), n_hat[s], n_del[s]);
  sp1[s] = make_float4(__double2float_ru(gamma * ((double)n_h[s] + (double)n_del[s])), one_f, 0.f, 0.f);
}

// max of {|vh|, |dv|} over each tile of 128 sorted items
__global__ void tile_norm_kernel(const float* __restrict__ n_h, const float* __restrict__ n_del, int n_items, int n_tiles, float2* __restrict__ out) {
  const int t = blockIdx.x, lane = threadIdx.x;   // 32 threads
  if (t >= n_tiles) return;
  float a = 0.f, b = 0.f;
  for (int i = t * kTN + lane; i < min(n_items, (t + 1) * kTN); i += 32) { a = fmaxf(a, n_h[i]); b = fmaxf(b, n_del[i]); }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) { a = fmaxf(a, __shfl_xor_sync(kFullMask, a, off)); b = fmaxf(b, __shfl_xor_sync(kFullMask, b, off)); }
  if (lane == 0) out[t] = make_float2(a, b);
}

// Item order: unsigned sort key that DESCENDS with |v|^2 (computed in fp64, compared as fp32 bit patterns of a
// non-negative float) and the identity permutation to sort along with it.
__global__ void item_sort_keys_kernel(const double* __restrict__ V, int K, int LD, int n, uint32_t* __restrict__ keys, int32_t* __restrict__ ids) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n) return;
  const double* x = V + (size_t)warp * LD;
  double s = 0.0;
  for (int k = lane; k < K; k += 32) s += x[k] * x[k];
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(kFullMask, s, off);
  if (lane == 0) {
    keys[warp] = ~__float_as_uint((float)s);   // larger norm -> smaller key -> earlier
    ids[warp] = warp;
  }
}

// flags[p] = 1 while the slot s at list position p stays in the working set: its certain count is below its limit,
// lim[s] (lim nullable: lim_all for every slot).  evaluate: topK + 1; ranking metrics: k + c_R per slot.
__global__ void below_limit_flags_kernel(const int32_t* __restrict__ list, const int32_t* __restrict__ n_list, int n_max,
                                         const int32_t* __restrict__ cnt_hi, const int32_t* __restrict__ lim, int lim_all,
                                         uint8_t* __restrict__ flags) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_max) return;
  const int n = n_list ? *n_list : n_max;
  uint8_t f = 0;
  if (p < n) {
    const int s = list ? list[p] : p;
    f = cnt_hi[s] < (lim ? lim[s] : lim_all);
  }
  flags[p] = f;
}

// W[p] = H[list[p]] (rows of KP halves, 16 bytes per thread)
__global__ void gather_rows_kernel(const __half* __restrict__ H, int KP, const int32_t* __restrict__ list, const int32_t* __restrict__ n_list,
                                   __half* __restrict__ W) {
  const int per_row = KP / 8;
  const long long n = (long long)(*n_list) * per_row;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x) {
    const int p = (int)(t / per_row), c = (int)(t % per_row);
    reinterpret_cast<uint4*>(W + (size_t)p * KP)[c] = __ldg(reinterpret_cast<const uint4*>(H + (size_t)list[p] * KP) + c);
  }
}

// ---- exact pass over the candidates -----------------------------------------------------------------
// One thread per pair: the reference's own score (sequential k, separately rounded products — predict(),
// MF_fastALS.cpp:208-221), compared with the exact gt score; (int)score kept for the ranking replay.
__global__ void __launch_bounds__(128)
eval_rescore_kernel(const double* __restrict__ U, const double* __restrict__ V, int K, int LD,
                    const int32_t* __restrict__ users, int u_begin, const double* __restrict__ gt_score,
                    EvalPair* __restrict__ pairs, const unsigned long long* __restrict__ n_pairs, unsigned long long cap,
                    int32_t* __restrict__ cnt_exact) {
  __shared__ double sm[4][2 * 32 * 17];
  const unsigned long long n = min(*n_pairs, cap);
  // whole warps stay in the loop together (seq_dot_warp32 is warp-cooperative)
  const unsigned long long n_round = (n + 31ull) & ~31ull;
  for (unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; t < n_round; t += (unsigned long long)gridDim.x * blockDim.x) {
    const bool live = t < n;
    EvalPair pr{0, 0, 0, 0};
    const double *a = nullptr, *b = nullptr;
    if (live) {
      pr = pairs[t];
      const int u = users ? users[pr.slot] : u_begin + pr.slot;
      a = U + (size_t)u * LD;
      b = V + (size_t)pr.item * LD;
    }
    const double acc = eals::seq_dot_warp32(a, b, K, sm[threadIdx.x >> 5]);
    if (live) {
      if ((pr.flags & 1) && acc > gt_score[pr.slot]) atomicAdd(cnt_exact + pr.slot, 1);
      pairs[t].key = __double2int_rz(acc);
    }
  }
}

}  // namespace tc
}  // namespace eals
