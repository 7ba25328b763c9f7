// cd_sweep.cuh — K1: the per-row coordinate-descent sweep of eALS.
//
// Replaces MF_fastALS::update_user_thread (MF_fastALS.cpp:243-322) and update_item_thread
// (:338-407).  For one row (a user, or an item on the transposed side) with nonzeros j = 1..n over
// neighbour rows y_j of the OTHER factor matrix, and the frozen S cache of the other side:
//
//   pred_j = <x, y_j>                                                      (:261-270 / :352-363)
//   for f = 0..K-1 (sequential — each step sees the factors updated before it):
//     numer = -g * sum_{k != f} x_k S[f][k]          g = 1 (user) | Wi[row] (item)   (:284-287 / :375-380)
//     pred_j -= x_f y_jf ; numer += (w_j r_j - c_j pred_j) y_jf ; denom += c_j y_jf^2     (:297-305 / :385-390)
//     denom += g S[f][f] + reg ;  x_f = numer / denom ; pred_j += x_f y_jf            (:307-315 / :391-400)
//   with c_j = w_j - Wi[item] (item = neighbour j on the user side, the row itself on the item side).
//
// Rows are independent inside a half-epoch (they only read the other side's factors, its S cache
// and Wi), so they are spread over warps / CTAs in any order; only the floating-point summation
// order over j differs from the reference's sequential loop.
//
// Data movement.  The n x K tile of gathered neighbour rows is what the K steps walk column by
// column.  It is staged through shared memory one 128-byte factor block (16 doubles of every
// gathered row = one full cache line each) at a time, so global memory sees whole lines exactly
// once per pass; the per-nonzero prediction cache lives in registers (warp kernel) or in a
// device-resident fp64 array (CTA kernel, rows of any length).
#pragma once

#include "common.cuh"

namespace eals {

// Replicas of the factor matrix being updated on the other GPUs of the box (CUDA IPC mappings of
// their X buffers): a finished row is stored straight into every replica over NVLink, which fuses
// the all-gather of the updated rows (SURVEY.md §8e, X2) into the sweep.
constexpr int kMaxPeers = 7;
struct PeerSet {
  double* x[kMaxPeers];
  int n;
};

struct CdSide {
  const int64_t* ptr;   // [rows+1] offsets of the owned rows (first owned row at 0)
  const int32_t* idx;   // neighbour ids, ascending inside a row
  const double* val;    // rating (= confidence weight) per nonzero, or nullptr for all-ones
  double* X;            // factors being updated, full replica [n][LD]
  const double* Y;      // the other side's factors [n'][LD]
  const double* S;      // the other side's S cache [K][LD]
  const double* Wi;     // item popularity weights [n_items]
  int row_base;         // global id of owned row 0
  int K;
  double reg;
  // Symmetric prediction cache.  The prediction <u, v> a user sweep leaves behind for a nonzero is
  // exactly the value the item sweep starts from (and vice versa), so the gather pass that rebuilds
  // it (MF_fastALS.cpp:261-270 / 352-363) is skipped: each side READS its own cache sequentially
  // (pc_in, this side's nonzero order) and WRITES local nonzero q's final prediction to pc_out[pc_map[q]].
  // One rank: pc_out is the other orientation's cache and pc_map the position of the same nonzero in it.
  // Several ranks: pc_out is a LOCAL staging array in destination order (pc_map: the slot in that order), and
  // the host copies each destination's segment to its owner afterwards.  Scattered 8-byte stores straight into
  // peer memory were far slower than the gather they replace (r01f).
  const double* pc_in;     // nullptr: no cache
  const uint32_t* pc_map;
  double* pc_out;          // nullptr: no cache output
  int use_cache;           // 1: pc_in is valid on entry, read it instead of recomputing
  PeerSet peers;        // other ranks' replicas of X (n = 0: none)
};

// No fence after the peer stores: grid completion already performs the kernel's stores at system scope before
// anything ordered after it in the stream (the event the other ranks wait on, or the NCCL all-reduce) can start.
// A per-thread __threadfence_system() cost 7 % at 4 GPUs (DESIGN.md §6).
__device__ __forceinline__ void store_row_value(const CdSide& a, size_t off, double v) {
  a.X[off] = v;
  for (int p = 0; p < a.peers.n; p++) a.peers.x[p][off] = v;
}

// The final prediction of a local nonzero, whose slot g = pc_map[local position] is already looked up.
__device__ __forceinline__ void pc_emit(const CdSide& a, uint32_t g, double v) { a.pc_out[g] = v; }

__device__ __forceinline__ void pc_store(const CdSide& a, int64_t local_pos, double v) {
  a.pc_out[a.pc_map[local_pos]] = v;
}

// inv[perm[k]] = k
__global__ void invert_perm_kernel(const uint32_t* __restrict__ perm, int64_t n, uint32_t* __restrict__ inv) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n) inv[perm[k]] = (uint32_t)k;
}

}  // namespace eals
