/* libtdvp_b200 -- C ABI of the B200-native TDVP hot path (complex128, sm_100a).
 *
 * The reference (PyTDSCF 1.3.3) has no FFI: its backend switch is a string ("numpy" | "jax") plus
 * duck-typed arrays (SURVEY.md 8(b)).  A `backend="cuda"` implements the narrow waist listed below by
 * calling these entry points through ctypes; each one names the reference interface it replaces
 * (file:line relative to the PyTDSCF tree).  INTEGRATION.md shows the reference-side binding.
 *
 * Conventions
 *   - every tensor argument is a DEVICE pointer to C-order complex128 (interleaved re,im), borrowed for the
 *     duration of the stream-ordered call; the library allocates only its own workspace;
 *   - every function returns int: 0 = OK, <0 = argument/shape/convergence error, >0 = CUDA error code;
 *     tdvp_last_error(handle) gives the message; nothing throws;
 *   - one handle per GPU / rank; calls on one handle are serialised by the caller; all work is enqueued on
 *     the handle's stream; the only host synchronisations are the scalar read-backs of the Krylov solver
 *     (alpha, beta, error per iteration) and of tdvp_inner;
 *   - index orders follow the reference: site tensor (D_l, d, D_r); environment block (bra, mpo, ket) =
 *     (D, w, D); full MPO core (w_l, d_bra, d_ket, w_r); diagonal MPO core (w_l, d, w_r).
 */
#ifndef TDVP_B200_H
#define TDVP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tdvp_handle_s* tdvp_handle_t;
typedef struct { double re, im; } tdvp_c128;

enum { TDVP_KIND_IDENTITY = 0, TDVP_KIND_DIAG = 3, TDVP_KIND_FULL = 4, TDVP_KIND_BLOCK = 3 };
enum { TDVP_KRYLOV_LANCZOS_REF = 0, TDVP_KRYLOV_ARNOLDI = 1 };
enum { TDVP_GAUGE_A = 0, TDVP_GAUGE_B = 1 };

/* One MPO term of H_eff (pytdscf/_contraction.py:1038-1176, `_op_lcr_dot`): (L, W, R) with identity
 * placeholders.  L: NULL (identity) or (Dl, wl, Dl).  W: NULL (identity; then wl == wr == 1), diagonal
 * (wl, d, wr) when w_kind == TDVP_KIND_DIAG, full (wl, d, d, wr) when TDVP_KIND_FULL.  R: NULL or
 * (Dr, wr, Dr).  `Wp` is an optional pre-permuted copy of a full core, Wp[c,j,i,t] = W[c,i,j,t]
 * (NULL: permuted on the fly).  `coef` scales the term (the reference's coupleJ on the "ovlp" term).
 * `id_channels` = (l_id + 1) | ((r_id + 1) << 16), 0 = none: optional promise by the caller that MPO channel l_id of L
 * (resp. r_id of R) is the identity matrix -- the "nothing happened yet / everything done" channel of an MPO whose
 * block was built from canonical (isometric) site tensors, where the reference contracts an explicit, numerically
 * unit block.  The library then copies instead of multiplying for that channel (large tensors only). */
typedef struct {
  const tdvp_c128* L;
  const tdvp_c128* W;
  const tdvp_c128* Wp;
  const tdvp_c128* R;
  int32_t wl, wr, w_kind, id_channels;
  double coef_re, coef_im;
} tdvp_heff_term;

/* One term of K_eff (pytdscf/_contraction.py:1297-1352, `_op_lr_dot`): L NULL or (D_l, w, D_l), R NULL or (D_r, w, D_r);
 * `id_channels` as in tdvp_heff_term. */
typedef struct {
  const tdvp_c128* L;
  const tdvp_c128* R;
  int32_t w, id_channels;
  double coef_re, coef_im;
} tdvp_keff_term;

/* ---- lifetime ---------------------------------------------------------------------------------- */
int tdvp_create(int device, void* cuda_stream, tdvp_handle_t* out);
int tdvp_destroy(tdvp_handle_t h);
const char* tdvp_last_error(tdvp_handle_t h);
int tdvp_abi_version(void);
/* counters: kernels launched by this library since load; Krylov solves / matvecs and algorithmic
 * contraction flops (SURVEY 8(d) formulas) issued through this handle */
unsigned long long tdvp_launch_count(void);
int tdvp_get_stats(tdvp_handle_t h, unsigned long long* solves, unsigned long long* matvecs, double* flops);
int tdvp_reset_stats(tdvp_handle_t h);
/* Per-launch CUDA-event timing of the DMMA ZGEMM kernel on its launching stream (bench.py roofline): collects what
 * was recorded so far into (ms, 8*M*N*K flops, launches), optionally resets the totals, then switches recording
 * on/off.  Synchronises on the recorded events. */
int tdvp_gemm_profile(int enable, int reset, double* ms, double* flops, unsigned long long* launches);
/* Per-label breakdown of everything recorded while profiling was on, as a JSON object written to `out`
 * (truncated to cap); returns the size needed. */
size_t tdvp_profile_json(char* out, size_t cap);

/* Test / tuning override of the GEMM launch choice for every later call on this handle (0 = automatic everywhere):
 * tile_cfg 1 = big (128x64 CTA tile), 2 = small (64x32), 3 = tiny (32x32), 4 = tma (persistent TMA-fed 128x64 with stream-K
 * balancing; shapes it cannot serve fall back to the automatic choice), 5 = tma with whole tiles only; splitk 1 = never split K, S >= 2 = S chunks where K allows;
 * c_stream 1 = always store C with evict-first, 2 = never.  The parity tests use it to pin EVERY configuration on the
 * benchmarked shapes (tests/test_gpu_bench_shapes.py); production code leaves it at 0. */
int tdvp_set_gemm_config(tdvp_handle_t h, int tile_cfg, int splitk, int c_stream);

/* ---- contractions ------------------------------------------------------------------------------ */
/* out(Dl,d,Dr) = sum_terms coef * L.W.R.psi  -- replaces multiplyH_MPS_direct_MPO.dot
 * (pytdscf/_contraction.py:1182-1243). */
int tdvp_heff_apply(tdvp_handle_t h, const tdvp_heff_term* terms, int nterms, int Dl, int d, int Dr,
                    const tdvp_c128* psi, tdvp_c128* out);
/* out(Dl,Dr) = sum_terms coef * L.sigma.R^T -- replaces multiplyK_MPS_direct_MPO.dot
 * (pytdscf/_contraction.py:1358-1407). */
int tdvp_keff_apply(tdvp_handle_t h, const tdvp_keff_term* terms, int nterms, int Dl, int Dr,
                    const tdvp_c128* sigma, tdvp_c128* out);
/* Environment update -- replaces contract_with_site_mpo (pytdscf/_contraction.py:148-397).
 * gauge A: out(Dr, w_out, Dr) from bra/ket (Dl,d,Dr), E NULL|(Dl,w_in,Dl), W as in tdvp_heff_term with
 *          (wl,wr) = (w_in,w_out);
 * gauge B: out(Dl, w_out, Dl) from bra/ket (Dl,d,Dr), E NULL|(Dr,w_in,Dr), W with (wl,wr) = (w_out,w_in).
 * `bra` is conjugated inside.  accumulate != 0 adds into `out` (the reference's "summed" blocks). */
int tdvp_env_update(tdvp_handle_t h, int gauge, int Dl, int d, int Dr, const tdvp_c128* bra,
                    const tdvp_c128* ket, const tdvp_c128* E, int w_in, const tdvp_c128* W, int w_kind,
                    int w_out, tdvp_c128* out, int accumulate);

/* ---- Krylov exponentials ----------------------------------------------------------------------- */
/* psi <- exp(scale * Op) psi with the reference's exact control flow (pytdscf/_integrator.py:453-655
 * short_iterative_lanczos, :287-432 short_iterative_arnoldi): alpha_l = <v0|Op v_l>, warm-up gating by
 * n_warmup, stop on |psi_k - psi_{k-1}| < thresh or beta < 1e-12 or k == size, conserve_norm handling.
 * Exactly one of (hterms, kterms) is non-NULL: H_eff on (Dl,d,Dr) or K_eff on (Dl,Dr) with d ignored.
 * niter receives the number of Krylov vectors used (the reference's _Debug.niter_krylov entry). */
/* Adaptive bond growth (pytdscf/_contraction.py:479-608 `stack(extend=True)` / `split(truncate=True)`): the next
 * tdvp_krylov_expm call runs on a zero-extended tensor but sizes its Krylov space (cap min(20, size), warm-up bound,
 * "space exhausted" test) by `size`, the number of elements of the tensor before extension, as the reference does
 * (pytdscf/_integrator.py:178-186).  One-shot: reset by the solve; 0 clears it. */
int tdvp_set_krylov_size(tdvp_handle_t h, long long size);
int tdvp_krylov_expm(tdvp_handle_t h, int kind, double scale_re, double scale_im, double thresh,
                     int n_warmup, int conserve_norm, const tdvp_heff_term* hterms,
                     const tdvp_keff_term* kterms, int nterms, int Dl, int d, int Dr,
                     tdvp_c128* psi_inout, int* niter);

/* psi <- normalised lowest (root == 0) or highest (root != 0) eigenvector of H_eff in the Krylov space grown from
 * psi by textbook Lanczos -- replaces matrix_diagonalize_lanczos (pytdscf/_integrator.py:74-138), the site solve of
 * improved relaxation.  The small tridiagonal eigenproblem is solved on device (bisection + inverse iteration); the
 * eigenvector sign is fixed to a positive overlap with the input (LAPACK's sign is unpinned in the reference). */
int tdvp_lanczos_eigvec(tdvp_handle_t h, const tdvp_heff_term* hterms, int nterms, int Dl, int d, int Dr,
                        tdvp_c128* psi_inout, int root, double thresh, int* niter);

/* ---- gauge shift ------------------------------------------------------------------------------- */
/* Householder QR with LAPACK zgeqrf/zungqr conventions -- replaces SiteCoef.gauge_trf
 * (pytdscf/_site_cls.py:138-292).  gauge A: psi(Dl,d,Dr) -> site(Dl,d,k), sigma(k,Dr);
 * gauge B: psi -> sigma(Dl,k), site(k,d,Dr); k = min(rows, cols) of the matricisation.  The row count has no limit
 * beyond the workspace: panels taller than num_sms x 256 rows keep their slabs in global memory. */
int tdvp_qr_shift(tdvp_handle_t h, int gauge, int Dl, int d, int Dr, const tdvp_c128* psi,
                  tdvp_c128* site, tdvp_c128* sigma);
/* gauge A: out(k,d,Dr) = sigma(k,Dl) . site(Dl,d,Dr);  gauge B: out(Dl,d,k) = site(Dl,d,Dr) . sigma(Dr,k)
 * -- replaces trans_next_psite_APsiB (pytdscf/_mps_cls.py:1172-1206). */
int tdvp_absorb(tdvp_handle_t h, int gauge, int Dl, int d, int Dr, int k, const tdvp_c128* sigma,
                const tdvp_c128* site, tdvp_c128* out);

/* ---- bond-matrix SVD (parallel / adaptive modes) --------------------------------------------------- */
/* SVD of the square bond matrix sigma(n,n) with the reference's truncation rule -- replaces truncate_sigvec
 * (pytdscf/_site_cls.py:586-690): keep the smallest idx with cumsum(s)[idx-1] / sum(s) >= 1 - p (singular VALUES,
 * not squares), optional flooring of small values (regularize: s + 1e-4 exp(-s/1e-4)), renormalised.
 * Outputs: U(n,n) and Vh(n,n) complete unitaries (leading *rank columns / rows are the kept ones), S = diag(s/|s|)
 * as a (k,k) matrix with k = n (keepdim, zero-padded) or k = *rank.  One-sided Jacobi on device; the truncation
 * decision reads the singular values back to the host. */
int tdvp_svd_truncate(tdvp_handle_t h, int m, int n, const tdvp_c128* sigma, double p, int keepdim, int regularize,
                      tdvp_c128* U, tdvp_c128* S, tdvp_c128* Vh, int* rank);
/* Thin SVD A(m,n) = U(m,n) diag(s) Vh(n,n), m >= n, s descending and written to HOST memory -- replaces
 * np.linalg.svd / scipy.linalg.svd in CC2ALambdaB (pytdscf/_mps_cls.py:3601-3630) and in the regularised gauge_trf
 * (pytdscf/_site_cls.py:207-252).  Any m >= n: zero singular values get their left vectors from a Householder QR,
 * which has no row limit (see tdvp_qr_shift). */
int tdvp_svd(tdvp_handle_t h, int m, int n, const tdvp_c128* A, tdvp_c128* U, double* s_host, tdvp_c128* Vh);
/* out(n,m) = pinv(X(m,n), rcond) -- replaces np.linalg.pinv in multiply_sigvec_pinv (pytdscf/_site_cls.py:734). */
int tdvp_pinv(tdvp_handle_t h, int m, int n, const tdvp_c128* X, double rcond, tdvp_c128* out);

/* ---- observables on device --------------------------------------------------------------------- */
/* <bra|ket> = sum conj(bra_i) ket_i (conj != 0) or sum bra_i ket_i  -- np.inner of
 * pytdscf/_integrator.py:65-71.  Result is written to host memory (synchronises the stream). */
int tdvp_inner(tdvp_handle_t h, long long n, const tdvp_c128* bra, const tdvp_c128* ket, int conj,
               tdvp_c128* host_out);
/* one site of the MPS overlap recursion block'(Dr_b,Dr_k) = sum bra[a,b,c] ket[i,b,k] block[a,i]
 * (pytdscf/wavefunction.py:248-255); conj_bra selects <Psi|Psi> vs the t/2-trick <Psi*|Psi>. */
int tdvp_overlap_site(tdvp_handle_t h, int Dlb, int Dlk, int d, int Drb, int Drk, const tdvp_c128* bra,
                      const tdvp_c128* ket, const tdvp_c128* block, int conj_bra, tdvp_c128* out);

/* ---- plain GEMM (exposed for tests / bench) ------------------------------------------------------ */
/* C(M,N) = alpha * op(A) . op(B) + beta * C, row-major; transX: 0 = N, 1 = T, 2 = C (conjugate transpose).
 * K = 0 gives C = beta * C (beta = 0: zeros, C is not read).  TDVP_ERR_ARG when lda, ldb or ldc is smaller than the
 * row length of its matrix as stored (A: K, or M when transposed; B: N, or K when transposed; C: N). */
int tdvp_zgemm(tdvp_handle_t h, int transA, int transB, int M, int N, int K, double alpha_re,
               double alpha_im, const tdvp_c128* A, int lda, const tdvp_c128* B, int ldb, double beta_re,
               double beta_im, tdvp_c128* C, int ldc);

#ifdef __cplusplus
}
#endif

/* two-site TDVP entry points (same conventions, same ABI version) */
#include "tdvp_b200_two_site.h"

#endif /* TDVP_B200_H */
