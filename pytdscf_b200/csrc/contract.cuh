#pragma once
#include "../../include/tdvp_b200.h"
#include "handle.cuh"

namespace tdvp {

// zgemm_auto on the handle's stream and GEMM context; a launch error is recorded on the handle as "CUDA error ... in <what>"
int gemm(Handle* h, const GemmDesc& g, const char* what = "zgemm_launch");

// workspace needs in complex128 elements (callers reserve before composing launches)
size_t heff_ws_elems(const tdvp_heff_term* terms, int nterms, int Dl, int d, int Dr);
size_t keff_ws_elems(const tdvp_keff_term* terms, int nterms, int Dl, int Dr);
size_t env_ws_elems(int Dl, int d, int Dr, int w_in, int w_out);

int heff_term_exec(Handle* h, const tdvp_heff_term& t, int Dl, int d, int Dr, const c128* psi, c128* out, bool accumulate);
int heff_apply_exec(Handle* h, const tdvp_heff_term* terms, int nterms, int Dl, int d, int Dr, const c128* psi, c128* out);
size_t heff2_ws_elems(const tdvp_heff2_term* terms, int nterms, int Dl, int d1, int d2, int Dr);
int heff2_term_exec(Handle* h, const tdvp_heff2_term& t, int Dl, int d1, int d2, int Dr, const c128* theta, c128* out,
                    bool accumulate);
int heff2_apply_exec(Handle* h, const tdvp_heff2_term* terms, int nterms, int Dl, int d1, int d2, int Dr, const c128* theta,
                     c128* out);
// ws_reserve that reports a request the device cannot hold as TDVP_ERR_NO_MEMORY with the size in the message
int ws_reserve_checked(Handle* h, size_t bytes, const char* what);
int keff_term_exec(Handle* h, const tdvp_keff_term& t, int Dl, int Dr, const c128* sigma, c128* out, bool accumulate);
int keff_apply_exec(Handle* h, const tdvp_keff_term* terms, int nterms, int Dl, int Dr, const c128* sigma, c128* out);
int env_update_exec(Handle* h, int gauge, int Dl, int d, int Dr, const c128* bra, const c128* ket, const c128* E,
                    int w_in, const c128* W, int w_kind, int w_out, c128* out, bool accumulate);
int overlap_site_exec(Handle* h, int Dlb, int Dlk, int d, int Drb, int Drk, const c128* bra, const c128* ket,
                      const c128* block, int conj_bra, c128* out);
int permute_site(Handle* h, const c128* in, c128* out, int Dl, int d, int Dr);

}  // namespace tdvp
