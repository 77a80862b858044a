/* libtdvp_b200 -- two-site TDVP entry points (complex128, sm_100a).
 *
 * Same conventions as tdvp_b200.h (device pointers to C-order complex128, int return codes, one handle per GPU), same
 * tdvp_abi_version(): these calls are additive.  A two-site tensor theta has the index order (D_l, d1, d2, D_r).
 * Return code -6 (TDVP_ERR_NO_MEMORY) means the device workspace could not grow to what the call needs; the message
 * of tdvp_last_error gives the requested size. */
#ifndef TDVP_B200_TWO_SITE_H
#define TDVP_B200_TWO_SITE_H

#include "tdvp_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

enum { TDVP_ERR_NO_MEMORY = -6 };

/* One MPO term of the two-site H_eff: (L, W1, W2, R) with identity placeholders.  L: NULL (identity; then wl == 1) or
 * (Dl, wl, Dl).  W1: NULL (identity; then wl == wm == 1), diagonal (wl, d1, wm) when w1_kind == TDVP_KIND_DIAG, full
 * (wl, d1, d1, wm) when TDVP_KIND_FULL.  W2 likewise with (wm, d2, wr).  R: NULL (then wr == 1) or (Dr, wr, Dr).
 * W1p / W2p: optional pre-permuted full cores as tdvp_heff_term's Wp (NULL: permuted on the fly).  A NULL core passes
 * a term that acts on only one of the two sites.  `coef` and `id_channels` (channel l_id of L, r_id of R) as in
 * tdvp_heff_term; the shortcut is taken for theta of at least 2^17 elements. */
typedef struct {
  const tdvp_c128* L;
  const tdvp_c128* W1;
  const tdvp_c128* W1p;
  const tdvp_c128* W2;
  const tdvp_c128* W2p;
  const tdvp_c128* R;
  int32_t wl, wm, wr, w1_kind, w2_kind, id_channels;
  double coef_re, coef_im;
} tdvp_heff2_term;

/* out(Dl,d1,d2,Dr)[a,i,k,r] = sum_terms coef * sum L[a,c,b] W1[c,i,j,t] W2[t,k,l,u] R[r,u,s] theta[b,j,l,s], contracted
 * L -> W1 -> W2 -> R as four stages on natural layouts (launch-profile labels heff2.s1 .. heff2.s4); `out` must not
 * alias `theta`. */
int tdvp_heff2_apply(tdvp_handle_t h, const tdvp_heff2_term* terms, int nterms, int Dl, int d1, int d2, int Dr,
                     const tdvp_c128* theta, tdvp_c128* out);

/* theta <- exp(scale * H2) theta, H2 the sum of the two-site terms, with the control flow of the one-site Krylov
 * exponential (same warm-up gating by n_warmup, stop rules, conserve_norm handling and Krylov cap min(20, size)).
 * The basis takes (k+1) Dl d1 d2 Dr complex128 elements of device memory; niter receives the Krylov dimension used. */
int tdvp_krylov_expm2(tdvp_handle_t h, int kind, double scale_re, double scale_im, double thresh, int n_warmup,
                      int conserve_norm, const tdvp_heff2_term* terms, int nterms, int Dl, int d1, int d2, int Dr,
                      tdvp_c128* theta_inout, int* niter);

/* Truncated split of a two-site tensor.  Thin SVD of the (Dl d1) x (d2 Dr) matricisation with the device Jacobi SVD
 * (through the conjugate transpose when Dl d1 < d2 Dr); rank r = min(r_p, Dcap) >= 1, r_p the smallest index with
 * cumsum(s)[r_p - 1] / sum(s) >= 1 - p (singular VALUES, the truncation rule of the bond SVD); Dcap is clipped to
 * min(Dl d1, d2 Dr).  conserve_norm != 0 scales the kept values by |s|_2 / |s_kept|_2, otherwise they stay as they are.
 *   direction TDVP_GAUGE_A: left = U[:, :r] (Dl,d1,r; gauge A), right = diag(s) Vh[:r] (r,d2,Dr; the centre);
 *   direction TDVP_GAUGE_B: left = U[:, :r] diag(s) (Dl,d1,r; the centre), right = Vh[:r] (r,d2,Dr; gauge B).
 * `left` / `right` are written densely with r columns / rows and must hold Dl d1 k and k d2 Dr elements for the clipped
 * k = Dcap.  s_host receives all min(Dl d1, d2 Dr) singular values, descending and unscaled: the rank is decided on
 * the host, one read-back per call. */
int tdvp_split2(tdvp_handle_t h, int direction, int Dl, int d1, int d2, int Dr, const tdvp_c128* theta, double p,
                int Dcap, int conserve_norm, tdvp_c128* left, tdvp_c128* right, double* s_host, int* rank);

#ifdef __cplusplus
}
#endif
#endif /* TDVP_B200_TWO_SITE_H */
