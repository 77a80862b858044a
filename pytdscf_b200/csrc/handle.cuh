// Per-GPU handle of libtdvp_b200: stream, error string, device workspace (bump allocator) and a
// pinned host mailbox for the few scalars the host control flow needs (Krylov alpha/beta/err).
#pragma once
#include "common.cuh"

#include <vector>

namespace tdvp {

struct Handle {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  // device workspace (grown on demand; calls on a handle are serialised by the caller)
  unsigned char* ws = nullptr;
  size_t ws_bytes = 0;
  size_t ws_top = 0;
  // small device scratch for reductions + pinned host mirror
  double* d_scal = nullptr;   // 4096 doubles
  double* h_scal = nullptr;   // pinned, 4096 doubles
  double* d_partial = nullptr;  // reduction partials: 1024 blocks x 64 doubles
  unsigned int* d_counter = nullptr;  // "last block done" tickets
  c128* d_splitk = nullptr;           // split-K partial products (SPLITK_SCRATCH_ELEMS)
  // side stream of the Krylov solver: the Ritz vector of the first checked iteration is formed there while the main
  // stream already runs the next matvec (own reduction partials / ticket, ordered against the main stream by events)
  cudaStream_t side = nullptr;
  cudaEvent_t ev_main = nullptr, ev_side = nullptr;
  double* d_partial_side = nullptr;
  unsigned int* d_counter_side = nullptr;
  GemmCtx gemm;                       // stream + scratch + overrides handed to every zgemm_auto call (gemm() in contract.cuh)
  // device limits queried once per handle (tdvp_create), never per process
  int num_sms = 148;
  int qr_max_cluster = 0;             // largest cluster the device co-schedules for k_qr_panel_cluster (0: none)
  int svd_max_blocks = 0;             // co-resident CTAs of k_jacobi_svd
  int svd_blocked_max_blocks = 0;     // co-resident CTAs of k_jacobi_svd_blocked (one per SM: it fills the shared memory)
  // statistics
  unsigned long long krylov_matvecs = 0;
  unsigned long long krylov_solves = 0;
  long long krylov_size_override = 0;   // > 0: size of the un-extended tensor (adaptive TDVP), consumed by the next solve
  double heff_flops = 0.0;  // algorithmic flops of H_eff/K_eff/env contractions issued (SURVEY 8(d) formulas)
};

// Make sure the workspace holds at least `bytes`; resets the bump pointer.
int ws_reserve(Handle* h, size_t bytes);
// Grow the workspace to at least `bytes` keeping its contents and the bump pointer (pointers into it move by the
// difference of the base addresses).
int ws_grow_preserve(Handle* h, size_t bytes);
// Bump allocation inside the reserved workspace (256-byte aligned). nullptr if it does not fit.
void* ws_alloc(Handle* h, size_t bytes);
inline void ws_reset(Handle* h) { h->ws_top = 0; }
inline size_t align256(size_t b) { return (b + 255) & ~size_t(255); }

}  // namespace tdvp
