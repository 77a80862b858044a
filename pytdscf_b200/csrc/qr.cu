// Blocked Householder QR with LAPACK zgeqrf / zungqr conventions for the TDVP gauge shift.
//
// Replaces scipy.linalg.qr(mode="economic") inside SiteCoef.gauge_trf (pytdscf/_site_cls.py:264-272, :279-291)
// and the sigma absorb of trans_next_psite_APsiB (pytdscf/_mps_cls.py:1187-1206).
//
// Why Householder with LAPACK's sign rule and not CholeskyQR/TSQR (SURVEY "hard parts"): the initial MPS is a
// Hartree product zero-padded to D, so early site tensors have EXACT zero columns; zlarfg returns tau = 0
// (identity reflector) for them and the null-space completion of Q is then a deterministic function of the
// leading reflectors.  One-site TDVP evolves inside the tangent space spanned by those completions, so the
// device QR reproduces zlarfg (beta = -sign(Re alpha)*norm, tau = (beta-alpha)/beta, v = x/(alpha-beta)),
// zlarft and the zlarfb block applications; only summation order differs from LAPACK.
//
// Panel factorisation (k_qr_panel): a cooperative kernel, one CTA per slab of <= SLAB_ROWS rows, the slab of
// the 32-column panel lives in shared memory for the whole panel.  A panel taller than num_sms x SLAB_ROWS rows gets
// one CTA per SM with ceil(rows / num_sms) rows each, and the slabs then live in a global-memory buffer instead.  Per column ONE grid-wide reduction gives
// both |x|^2 and every v^H a_j: with g_j = sum_{i>c} conj(a_ic) a_ij,  w_j = a_cj + conj(s) g_j where
// s = 1/(alpha - beta).  Partials are combined in fixed CTA order (deterministic).  Trailing updates and the
// formation of Q are DMMA ZGEMMs on explicit unit-lower-trapezoidal V panels.
#include <cooperative_groups.h>

#include "contract.cuh"

namespace cg = cooperative_groups;

namespace tdvp {

namespace {

constexpr int NB = 32;           // panel width
constexpr int SLAB_ROWS = 256;   // rows of the panel held per CTA (256*32*16 B = 128 KiB)
constexpr int PT = 256;          // threads per CTA, arranged (32, 8)
constexpr int PTY = PT / 32;

struct PanelArgs {
  c128* A; int lda; int m; int n; int j0; int jb;
  double* tau;     // complex tau per column of the whole matrix (2 doubles each)
  c128* Vall;      // explicit V, same shape as A (ld = lda)
  c128* Tall;      // per panel NB x NB upper triangular T (row-major), panel p at Tall + p*NB*NB
  double* gpart;   // 2 buffers x G x (2*NB complex): [buf][cta][0..NB) partial g, [NB..2NB) diagonal row broadcast
  double* zpart;   // G x NB x NB complex partial Gram for T
  int rows_per_cta;
  c128* gslab;     // k_qr_panel only: nullptr = slabs in shared memory, else [G][rows_per_cta][NB] in global memory
  int dbg;         // timing experiments only (TDVP_QR_DEBUG): bit 0 skips the column loop, bit 1 the T factor
};

__device__ __forceinline__ double dlapy3(double x, double y, double z) {
  const double w = fmax(fabs(x), fmax(fabs(y), fabs(z)));
  if (w == 0.0) return 0.0;
  const double a = x / w, b = y / w, c = z / w;
  return w * sqrt(a * a + b * b + c * c);
}

__global__ void __launch_bounds__(PT, 1) k_qr_panel(PanelArgs p) {
  extern __shared__ __align__(16) unsigned char smraw[];
  // [rows_per_cta][NB]; only this CTA touches its slab, so __syncthreads orders the global-memory variant too
  c128* S = p.gslab ? p.gslab + (size_t)blockIdx.x * p.rows_per_cta * NB : reinterpret_cast<c128*>(smraw);
  __shared__ c128 red[PTY][NB];
  __shared__ c128 gtot[NB];     // reduced g_j
  __shared__ c128 rowc[NB];     // row c of the panel (broadcast)
  __shared__ c128 wv[NB];       // w_j
  __shared__ double s_tau[2], s_scal[2], s_beta;
  cg::grid_group grid = cg::this_grid();
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int G = gridDim.x, b = blockIdx.x;
  const int jb = p.jb, j0 = p.j0;
  const int r0 = j0 + b * p.rows_per_cta;                   // first global row of this slab
  int nrow = p.m - r0;
  if (nrow > p.rows_per_cta) nrow = p.rows_per_cta;
  if (nrow < 0) nrow = 0;

  // ---- load slab ----
  for (int i = ty; i < nrow; i += PTY) {
    if (tx < jb) S[i * NB + tx] = p.A[(long long)(r0 + i) * p.lda + j0 + tx];
    else S[i * NB + tx] = {0.0, 0.0};
  }
  __syncthreads();

  for (int c = 0; c < jb; ++c) {
    const int grow = j0 + c;                                 // global row of the diagonal element
    double* gp = p.gpart + (size_t)(c & 1) * G * (4 * NB);
    // (a) partial g_j = sum_{rows > grow} conj(a_ic) a_ij   for j = tx >= c
    c128 acc = {0.0, 0.0};
    if (tx >= c && tx < jb) {
      for (int i = ty; i < nrow; i += PTY) {
        if (r0 + i > grow) {
          const c128 x = S[i * NB + c], y = S[i * NB + tx];
          acc.x += x.x * y.x + x.y * y.y;
          acc.y += x.x * y.y - x.y * y.x;
        }
      }
    }
    red[ty][tx] = acc;
    __syncthreads();
    if (ty == 0) {
      c128 t = {0.0, 0.0};
#pragma unroll
      for (int q = 0; q < PTY; ++q) { t.x += red[q][tx].x; t.y += red[q][tx].y; }
      gp[(size_t)b * (4 * NB) + 2 * tx] = t.x;
      gp[(size_t)b * (4 * NB) + 2 * tx + 1] = t.y;
      // owner of the diagonal row broadcasts it
      if (grow >= r0 && grow < r0 + nrow) {
        const c128 v = S[(grow - r0) * NB + tx];
        gp[2 * NB + 2 * tx] = v.x;          // slot of CTA 0, upper half: shared broadcast area
        gp[2 * NB + 2 * tx + 1] = v.y;
      }
    }
    __threadfence();
    if (G > 1) grid.sync(); else __syncthreads();
    // (c) total g and the diagonal row
    if (ty == 0) {
      c128 t = {0.0, 0.0};
      for (int q = 0; q < G; ++q) {
        t.x += __ldcg(&gp[(size_t)q * (4 * NB) + 2 * tx]);
        t.y += __ldcg(&gp[(size_t)q * (4 * NB) + 2 * tx + 1]);
      }
      gtot[tx] = t;
      rowc[tx] = {__ldcg(&gp[2 * NB + 2 * tx]), __ldcg(&gp[2 * NB + 2 * tx + 1])};
    }
    __syncthreads();
    // (d) zlarfg
    if (tx == 0 && ty == 0) {
      // |x|^2 below 1e-200 cannot be formed accurately as a plain sum of squares (the terms are denormal); LAPACK's
      // dznrm2 rescales, here such a tail (|x| < 1e-100 next to O(1) data) is treated as exactly zero: the reflector
      // degenerates to a phase on the diagonal and Q stays an isometry to rounding.
      const bool tiny_tail = gtot[c].x < 1.0e-200;
      const double xnorm = tiny_tail ? 0.0 : sqrt(gtot[c].x);
      const double alphr = rowc[c].x, alphi = rowc[c].y;
      if (xnorm == 0.0 && alphi == 0.0) {
        s_tau[0] = 0.0; s_tau[1] = 0.0; s_scal[0] = 1.0; s_scal[1] = 0.0; s_beta = alphr;
      } else if (tiny_tail) {
        const double beta = (alphr >= 0.0) ? -hypot(alphr, alphi) : hypot(alphr, alphi);
        s_tau[0] = (beta - alphr) / beta;
        s_tau[1] = -alphi / beta;
        s_scal[0] = 0.0; s_scal[1] = 0.0;                    // v = e_1: the tail is dropped
        s_beta = beta;
      } else {
        double beta = dlapy3(alphr, alphi, xnorm);
        beta = (alphr >= 0.0) ? -beta : beta;               // -SIGN(norm, alphr)
        s_tau[0] = (beta - alphr) / beta;
        s_tau[1] = -alphi / beta;
        // s = 1 / (alpha - beta)   (zladiv)
        const double dr = alphr - beta, di = alphi;
        const double den = dr * dr + di * di;
        s_scal[0] = dr / den; s_scal[1] = -di / den;
        s_beta = beta;
      }
      if (b == 0) { p.tau[2 * (j0 + c)] = s_tau[0]; p.tau[2 * (j0 + c) + 1] = s_tau[1]; }
    }
    __syncthreads();
    const c128 tau = {s_tau[0], s_tau[1]};
    const c128 sc = {s_scal[0], s_scal[1]};
    const bool trivial = (tau.x == 0.0 && tau.y == 0.0);
    if (ty == 0 && tx > c && tx < jb) {
      // w_j = a_cj + conj(s) g_j
      const c128 cs = {sc.x, -sc.y};
      wv[tx] = cadd(rowc[tx], cmul(cs, gtot[tx]));
    }
    __syncthreads();
    // (e) scale x, apply H^H = I - conj(tau) v v^H to the remaining panel columns, set the diagonal
    if (!trivial) {
      const c128 ctau = {tau.x, -tau.y};
      for (int i = ty; i < nrow; i += PTY) {
        const int gr = r0 + i;
        if (gr < grow) continue;
        c128 v;
        if (gr == grow) v = {1.0, 0.0};
        else v = cmul(S[i * NB + c], sc);
        if (tx > c && tx < jb) {
          const c128 f = cmul(ctau, cmul(v, wv[tx]));
          S[i * NB + tx].x -= f.x;
          S[i * NB + tx].y -= f.y;
        }
        __syncwarp();
        if (tx == c) S[i * NB + c] = (gr == grow) ? c128{s_beta, 0.0} : v;
      }
    }
    __syncthreads();
  }

  // ---- write back: R / v into A, explicit V into Vall, partial Gram Z = V^H V for T ----
  for (int i = ty; i < nrow; i += PTY) {
    const int gr = r0 + i;
    if (tx < jb) {
      const c128 a = S[i * NB + tx];
      p.A[(long long)gr * p.lda + j0 + tx] = a;
      c128 v;
      const int dcol = gr - j0;                              // column whose diagonal sits in this row
      if (tx < dcol) v = a;
      else if (tx == dcol) v = {1.0, 0.0};
      else v = {0.0, 0.0};
      p.Vall[(long long)gr * p.lda + j0 + tx] = v;
      S[i * NB + tx] = v;
    }
  }
  __syncthreads();
  // Z[a, c] = sum_i conj(V[i,a]) V[i,c], a < c: thread (ty, tx) owns column c = tx, rows a = ty, ty+8, ...
  for (int a = ty; a < jb; a += PTY) {
    c128 z = {0.0, 0.0};
    if (tx < jb && a < tx) {
      for (int i = 0; i < nrow; ++i) {
        const c128 x = S[i * NB + a], y = S[i * NB + tx];
        z.x += x.x * y.x + x.y * y.y;
        z.y += x.x * y.y - x.y * y.x;
      }
    }
    p.zpart[((size_t)b * NB + a) * NB * 2 + 2 * tx] = z.x;
    p.zpart[((size_t)b * NB + a) * NB * 2 + 2 * tx + 1] = z.y;
  }
  __threadfence();
  if (G > 1) grid.sync(); else __syncthreads();
  if (b != 0) return;
  // ---- T (zlarft, forward/columnwise) by CTA 0 ----
  c128* Z = S;               // reuse: [NB][NB]
  c128* T = S + NB * NB;
  for (int a = ty; a < NB; a += PTY) {
    c128 z = {0.0, 0.0};
    for (int q = 0; q < G; ++q) {
      z.x += __ldcg(&p.zpart[((size_t)q * NB + a) * NB * 2 + 2 * tx]);
      z.y += __ldcg(&p.zpart[((size_t)q * NB + a) * NB * 2 + 2 * tx + 1]);
    }
    Z[a * NB + tx] = z;
    T[a * NB + tx] = {0.0, 0.0};
  }
  __syncthreads();
  for (int c = 0; c < jb; ++c) {
    const c128 tau = {__ldcg(&p.tau[2 * (j0 + c)]), __ldcg(&p.tau[2 * (j0 + c) + 1])};
    // T[0:c, c] = -tau * T[0:c, 0:c] @ Z[0:c, c]
    if (ty == 0 && tx < c) {
      c128 s = {0.0, 0.0};
      for (int q = tx; q < c; ++q) s = cadd(s, cmul(T[tx * NB + q], Z[q * NB + c]));
      const c128 r = cmul(tau, s);
      T[tx * NB + c] = {-r.x, -r.y};
    }
    if (ty == 0 && tx == c) T[c * NB + c] = tau;
    __syncthreads();
  }
  c128* Tout = p.Tall + (size_t)(j0 / NB) * NB * NB;
  for (int a = ty; a < NB; a += PTY) Tout[a * NB + tx] = T[a * NB + tx];
}


// ---- cluster variant: the whole panel is owned by ONE thread-block cluster (<= 16 CTAs).  Same arithmetic and the same
// fixed CTA-order summation as k_qr_panel, but the per-column exchange is a PUSH through distributed shared memory:
// every CTA stores its 32 partial inner products (and the owner of the diagonal row that row) straight into the inbox of
// every CTA of the cluster with st.async, which also counts the bytes on the receiver's mbarrier.  A CTA then waits on
// its OWN barrier and reads its OWN shared memory -- no cluster-wide hardware barrier and no remote-load round trip per
// column (r1: cluster.sync + DSMEM gather + zlarfg's division chain = ~5 us per column, a third of it barrier wait). ----
constexpr int CT = 512;           // threads per CTA, arranged (32, 16): 128 registers per thread for the resident slab
constexpr int CTY = CT / 32;
constexpr int MAXG = 16;          // largest cluster
constexpr int CL_ROWS = 256;     // slab rows per CTA in the cluster kernel: 16 rows per thread in registers, 128 KiB staged in shared memory

__device__ __forceinline__ unsigned qr_smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ unsigned qr_mapa(unsigned local, int cta) {
  unsigned r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(r) : "r"(local), "r"(cta));
  return r;
}
__device__ __forceinline__ void qr_push(unsigned remote_addr, c128 v, unsigned remote_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f64 [%0], {%1, %2}, [%3];\n" ::"r"(remote_addr),
               "d"(v.x), "d"(v.y), "r"(remote_bar)
               : "memory");
}
__device__ __forceinline__ bool qr_try_wait(unsigned bar, unsigned parity) {
  unsigned ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.b32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}

// zlarfg scalars of one column: tau, s = 1 / (alpha - beta), beta, from alpha = (alphr, alphi) and g2 = |x|^2 of the
// entries below the diagonal.  LAPACK forms the norm with dlapy3's scaled sum (3 divisions + sqrt) and the reciprocal with
// zladiv; in the range where nothing can overflow or underflow the plain forms give the same values to rounding with one
// sqrt and two reciprocals (the FP64 division chain was a third of the panel's per-column latency).
__device__ __forceinline__ void zlarfg_scalars(double alphr, double alphi, double g2, c128& tau, c128& sc, double& hbeta) {
  // |x|^2 below 1e-200 cannot be formed accurately as a plain sum of squares (the terms are denormal); LAPACK's
  // dznrm2 rescales, here such a tail (|x| < 1e-100 next to O(1) data) is treated as exactly zero: the reflector
  // degenerates to a phase on the diagonal and Q stays an isometry to rounding.
  const bool tiny_tail = g2 < 1.0e-200;
  if (tiny_tail && alphi == 0.0) { tau = {0.0, 0.0}; sc = {1.0, 0.0}; hbeta = alphr; return; }   // H = I (zlarfg: tau = 0)
  if (tiny_tail) {
    const double beta = (alphr >= 0.0) ? -hypot(alphr, alphi) : hypot(alphr, alphi);
    tau = {(beta - alphr) / beta, -alphi / beta};
    sc = {0.0, 0.0};                                    // v = e_1: the tail is dropped
    hbeta = beta;
    return;
  }
  double beta;
  if (g2 < 1.0e280 && fabs(alphr) < 1.0e140 && fabs(alphi) < 1.0e140) beta = sqrt(alphr * alphr + alphi * alphi + g2);   // g2 >= 1e-200 here
  else beta = dlapy3(alphr, alphi, sqrt(g2));
  beta = (alphr >= 0.0) ? -beta : beta;                 // -SIGN(norm, alphr)
  const double rb = 1.0 / beta;
  tau = {(beta - alphr) * rb, -alphi * rb};
  const double dr = alphr - beta, di = alphi;
  const double rd = 1.0 / (dr * dr + di * di);           // s = 1 / (alpha - beta)
  sc = {dr * rd, -di * rd};
  hbeta = beta;
}

__global__ void __launch_bounds__(CT, 1) k_qr_panel_cluster(PanelArgs p) {
  extern __shared__ __align__(16) unsigned char smraw[];
  c128* S = reinterpret_cast<c128*>(smraw);                 // [rows_per_cta][NB]
  __shared__ c128 red[CTY][NB + 1];
  __shared__ __align__(16) c128 inbox[2][MAXG + 1][NB];     // [column parity][source CTA | MAXG: diagonal row][panel column]
  __shared__ __align__(8) unsigned long long mbar[2];
  __shared__ c128 gtot[NB], rowc[NB], rowstage[NB];
  __shared__ double s_zl[5];     // zlarfg scalars of the current column: tau, 1/(alpha - beta), beta
  cg::cluster_group cluster = cg::this_cluster();
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int G = gridDim.x, b = blockIdx.x;                   // the grid is exactly one cluster: rank == blockIdx.x
  const int jb = p.jb, j0 = p.j0;
  const int r0 = j0 + b * p.rows_per_cta;
  int nrow = p.m - r0;
  if (nrow > p.rows_per_cta) nrow = p.rows_per_cta;
  if (nrow < 0) nrow = 0;

  if (tx == 0 && ty == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(qr_smem_u32(&mbar[0])) : "memory");
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(qr_smem_u32(&mbar[1])) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  for (int i = ty; i < nrow; i += CTY) {
    if (tx < jb) S[i * NB + tx] = p.A[(long long)(r0 + i) * p.lda + j0 + tx];
    else S[i * NB + tx] = {0.0, 0.0};
  }
  __syncthreads();
  cluster.sync();                                            // every inbox barrier exists before the first remote push

  // The slab lives in REGISTERS during the column loop: thread (tx, ty) owns column tx of the rows ty, ty + 32, ... of this
  // CTA (at most MAXPER of them).  A warp is one row group, its lanes are the 32 panel columns, so the column-c entries a
  // thread needs for its own rows sit in lane c of the SAME warp: one shuffle instead of a shared-memory round trip per
  // row (r2 ncu: the slab pass through shared memory was 44 % of the kernel's samples, MIO-bound).
  constexpr int MAXPER = (CL_ROWS + CTY - 1) / CTY;
  c128 mine[MAXPER];
#pragma unroll
  for (int k = 0; k < MAXPER; ++k) {
    const int i = ty + CTY * k;
    mine[k] = (i < nrow) ? S[i * NB + tx] : c128{0.0, 0.0};
  }
  // partial g for column 0; for c > 0 it is accumulated while column c-1 is applied (one pass over the slab per column)
  c128 acc = {0.0, 0.0};
#pragma unroll
  for (int k = 0; k < MAXPER; ++k) {
    const int i = ty + CTY * k;
    const double xr = __shfl_sync(0xffffffffu, mine[k].x, 0), xi = __shfl_sync(0xffffffffu, mine[k].y, 0);
    if (i < nrow && r0 + i > j0 && tx < jb) {
      acc.x += xr * mine[k].x + xi * mine[k].y;
      acc.y += xr * mine[k].y - xi * mine[k].x;
    }
    if (i < nrow && r0 + i == j0) rowstage[tx] = mine[k];     // diagonal row of column 0, staged for its owner's push
  }
  for (int c = 0; c < ((p.dbg & 1) ? 0 : jb); ++c) {
    const int grow = j0 + c;
    const int buf = c & 1;
    const unsigned parity = (unsigned)(c >> 1) & 1u;
    const int owner = c / p.rows_per_cta;
    red[ty][tx] = acc;
    __syncthreads();                                          // (rowstage holds row `grow`: staged by the previous pass)
    {
      // warp ty reduces columns ty (lanes 0-15) and ty + 16 (lanes 16-31) over the 16 row groups (fixed butterfly order:
      // every lane of a half ends up with the total) and lane q of each half pushes it into CTA q's inbox; warps 0..G-1 of
      // the diagonal row's owner also push that row, one CTA each
      const int half = tx >> 4, q = tx & 15, col = ty + CTY * half;
      c128 t = red[q][col];
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) {
        t.x += __shfl_xor_sync(0xffffffffu, t.x, o);
        t.y += __shfl_xor_sync(0xffffffffu, t.y, o);
      }
      const unsigned bar_local = qr_smem_u32(&mbar[buf]);
      if (q < G) qr_push(qr_mapa(qr_smem_u32(&inbox[buf][b][col]), q), t, qr_mapa(bar_local, q));
      if (b == owner && ty < G) qr_push(qr_mapa(qr_smem_u32(&inbox[buf][MAXG][tx]), ty), rowstage[tx], qr_mapa(bar_local, ty));
    }
    if (ty == 0) {
      const unsigned bar = qr_smem_u32(&mbar[buf]);
      if (tx == 0) {
        const unsigned bytes = (unsigned)((G + 1) * NB * sizeof(c128));
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
      }
      __syncwarp();
      while (!qr_try_wait(bar, parity)) {
      }
      c128 t = {0.0, 0.0};
#pragma unroll
      for (int q = 0; q < MAXG; ++q) {
        if (q < G) { const c128 v = inbox[buf][q][tx]; t.x += v.x; t.y += v.y; }
      }
      const c128 rc = inbox[buf][MAXG][tx];
      gtot[tx] = t;
      rowc[tx] = rc;
      // zlarfg by this warp (every lane the same values), published through shared memory
      const double g2 = __shfl_sync(0xffffffffu, t.x, c);
      const double alphr = __shfl_sync(0xffffffffu, rc.x, c), alphi = __shfl_sync(0xffffffffu, rc.y, c);
      c128 tau_, sc_;
      double hb_;
      zlarfg_scalars(alphr, alphi, g2, tau_, sc_, hb_);
      if (tx == 0) {
        s_zl[0] = tau_.x; s_zl[1] = tau_.y; s_zl[2] = sc_.x; s_zl[3] = sc_.y; s_zl[4] = hb_;
        if (b == 0) { p.tau[2 * (j0 + c)] = tau_.x; p.tau[2 * (j0 + c) + 1] = tau_.y; }
      }
    }
    __syncthreads();
    const c128 tau = {s_zl[0], s_zl[1]}, sc = {s_zl[2], s_zl[3]};
    const double hbeta = s_zl[4];
    const bool trivial = (tau.x == 0.0 && tau.y == 0.0);
    // a_ij -= conj(tau) v_i w_j with v_i = s a_ic (v = 1 on the diagonal row), w_j = a_cj + conj(s) g_j.  The products
    // that do not depend on the row are formed once per column and thread: y_j = conj(tau) s w_j (rows below the
    // diagonal) and yd_j = conj(tau) w_j (diagonal row); the slab pass then costs one complex multiply-add per element.
    c128 yj = {0.0, 0.0}, ydj = {0.0, 0.0};
    if (tx > c && tx < jb) {
      const c128 cs = {sc.x, -sc.y};
      const c128 wv = cadd(rowc[tx], cmul(cs, gtot[tx]));
      const c128 ctau = {tau.x, -tau.y};
      ydj = cmul(ctau, wv);
      yj = cmul(sc, ydj);
    }
    // apply H^H to the remaining columns, store v / beta in column c, and in the same pass accumulate the next column's
    // partial g (lane c+1 holds the freshly updated a_{i,c+1})
    acc = {0.0, 0.0};
    const int cn = (c + 1 < NB) ? c + 1 : c;
#pragma unroll
    for (int k = 0; k < MAXPER; ++k) {
      const int i = ty + CTY * k;
      const int gr = r0 + i;
      // uniform per warp: ty and k select the row (shuffles below are executed by all lanes of the warp or by none)
      if (i >= nrow || gr < grow) continue;
      if (!trivial) {
        const double xr = __shfl_sync(0xffffffffu, mine[k].x, c), xi = __shfl_sync(0xffffffffu, mine[k].y, c);
        const c128 x = {xr, xi};
        if (tx > c && tx < jb) {
          const c128 f = (gr == grow) ? ydj : cmul(x, yj);
          mine[k].x -= f.x;
          mine[k].y -= f.y;
        }
        if (tx == c) mine[k] = (gr == grow) ? c128{hbeta, 0.0} : cmul(x, sc);
      }
      const double nr = __shfl_sync(0xffffffffu, mine[k].x, cn);
      const double ni = __shfl_sync(0xffffffffu, mine[k].y, cn);
      if (gr > grow + 1 && tx > c && tx < jb) {
        acc.x += nr * mine[k].x + ni * mine[k].y;
        acc.y += nr * mine[k].y - ni * mine[k].x;
      }
      if (gr == grow + 1) rowstage[tx] = mine[k];             // the next column's diagonal row, now final: staged for its push
    }
  }
  // back to shared memory for the write-back, the explicit V and the Gram matrix of the T factor
#pragma unroll
  for (int k = 0; k < MAXPER; ++k) {
    const int i = ty + CTY * k;
    if (i < nrow) S[i * NB + tx] = mine[k];
  }
  __syncthreads();

  for (int i = ty; i < nrow; i += CTY) {
    const int gr = r0 + i;
    if (tx < jb) {
      const c128 a = S[i * NB + tx];
      p.A[(long long)gr * p.lda + j0 + tx] = a;
      c128 v;
      const int dcol = gr - j0;
      if (tx < dcol) v = a;
      else if (tx == dcol) v = {1.0, 0.0};
      else v = {0.0, 0.0};
      p.Vall[(long long)gr * p.lda + j0 + tx] = v;
      S[i * NB + tx] = v;
    }
  }
  __syncthreads();
  // partial Gram Z[a, c] = sum_i conj(V[i,a]) V[i,c] (a < c), rows a = ty, ty + 16, column c = tx; kept in global scratch
  for (int a = ty; a < NB; a += CTY) {
    c128 z = {0.0, 0.0};
    if (tx < jb && a < tx) {
      for (int i = 0; i < nrow; ++i) {
        const c128 x = S[i * NB + a], y = S[i * NB + tx];
        z.x += x.x * y.x + x.y * y.y;
        z.y += x.x * y.y - x.y * y.x;
      }
    }
    p.zpart[((size_t)b * NB + a) * NB * 2 + 2 * tx] = z.x;
    p.zpart[((size_t)b * NB + a) * NB * 2 + 2 * tx + 1] = z.y;
  }
  __threadfence();
  cluster.sync();
  if (b != 0) return;
  // ---- T (zlarft, forward / columnwise) by CTA 0.  Row r of T depends only on row r itself:
  // T[r][c] = -tau_c sum_{q = r}^{c-1} T[r][q] Z[q][c], so lane r of ONE warp builds its row without any barrier
  // (T is kept transposed in shared memory: lanes read consecutive addresses, Z[q][c] is a broadcast). ----
  c128* Z = S;
  c128* Tt = S + NB * NB;        // Tt[q * NB + r] = T[r][q]
  __shared__ c128 taus[NB];
  for (int a = ty; a < NB; a += CTY) {
    c128 z = {0.0, 0.0};
    for (int q = 0; q < G; ++q) {
      z.x += __ldcg(&p.zpart[((size_t)q * NB + a) * NB * 2 + 2 * tx]);
      z.y += __ldcg(&p.zpart[((size_t)q * NB + a) * NB * 2 + 2 * tx + 1]);
    }
    Z[a * NB + tx] = z;
    Tt[a * NB + tx] = {0.0, 0.0};
    if (a == 0) taus[tx] = (tx < jb) ? c128{__ldcg(&p.tau[2 * (j0 + tx)]), __ldcg(&p.tau[2 * (j0 + tx) + 1])} : c128{0.0, 0.0};
  }
  __syncthreads();
  if (ty == 0 && !(p.dbg & 2)) {
    const int r = tx;
    if (r < jb) {
      Tt[r * NB + r] = taus[r];
      for (int c = r + 1; c < jb; ++c) {
        c128 s0 = {0.0, 0.0}, s1 = {0.0, 0.0};
        int q = r;
        for (; q + 1 < c; q += 2) {
          const c128 a0 = Tt[q * NB + r], z0 = Z[q * NB + c];
          const c128 a1 = Tt[(q + 1) * NB + r], z1 = Z[(q + 1) * NB + c];
          s0.x += a0.x * z0.x - a0.y * z0.y; s0.y += a0.x * z0.y + a0.y * z0.x;
          s1.x += a1.x * z1.x - a1.y * z1.y; s1.y += a1.x * z1.y + a1.y * z1.x;
        }
        if (q < c) {
          const c128 a0 = Tt[q * NB + r], z0 = Z[q * NB + c];
          s0.x += a0.x * z0.x - a0.y * z0.y; s0.y += a0.x * z0.y + a0.y * z0.x;
        }
        const c128 rr = cmul(taus[c], cadd(s0, s1));
        Tt[c * NB + r] = {-rr.x, -rr.y};
      }
    }
  }
  __syncthreads();
  c128* Tout = p.Tall + (size_t)(j0 / NB) * NB * NB;
  for (int a = ty; a < NB; a += CTY) Tout[a * NB + tx] = Tt[tx * NB + a];
}

__global__ void k_set_identity(c128* Q, int m, int n, int ld) {
  const long long tot = (long long)m * n;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x) {
    const int i = e / n, j = e % n;
    Q[(long long)i * ld + j] = {i == j ? 1.0 : 0.0, 0.0};
  }
}

__global__ void k_extract_r(const c128* A, int lda, int k, int n, c128* R, int ldr, int transpose) {
  // R (k x n upper trapezoidal) from A; transpose != 0 writes R^T (n x k, ld = ldr)
  const long long tot = (long long)k * n;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x) {
    const int i = e / n, j = e % n;
    const c128 v = (j >= i) ? A[(long long)i * lda + j] : c128{0.0, 0.0};
    if (transpose) R[(long long)j * ldr + i] = v; else R[(long long)i * ldr + j] = v;
  }
}

// W(jb x nc, ld = nc) = V^H C for a tall panel V (mp x jb, ld = ldv) and C (mp x nc, ld = ldc), issued as the
// transposed product W^T = C^T conj(V) so that the long dimension nc maps to the 128-row tile direction and the
// reduction over the mp rows is split across CTAs (split-K) instead of running on a handful of SMs.
GemmDesc vhc_desc(int jb, int nc, int mp, const c128* V, long long ldv, const c128* C, long long ldc, c128* W, const char* tag) {
  GemmDesc g;
  g.M = nc; g.N = jb; g.K = mp;
  g.A = C; g.a_m_inner = 1; g.a_m1 = 1; g.a_m0 = 0; g.a_k = ldc; g.a_conj = 0;
  g.B = V; g.b_n_inner = 1; g.b_n1 = 1; g.b_n0 = 0; g.b_k = ldv; g.b_conj = 1;
  g.C = W; g.c_m_inner = 1; g.c_m1 = 1; g.c_m0 = 0; g.c_n = nc;
  g.tag = tag;
  return g;
}

int lq(Handle* h, const char* what) {
  count_launch();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(h, e, what, __FILE__, __LINE__);
  return 0;
}

}  // namespace

constexpr int QR_MAX_SMS = 256;  // workspace bound for the per-CTA partials (B200: 148 SMs)

size_t qr_ws_elems(int m, int n) {
  const size_t np = (n + NB - 1) / NB;
  return 3 * (size_t)m * n + (size_t)(m + QR_MAX_SMS) * NB + np * NB * NB + 2 * (size_t)NB * n + 4096 + (size_t)QR_MAX_SMS * NB * NB + QR_MAX_SMS * 4 * NB;
}

// Per-device kernel attributes and co-scheduling limits of the panel kernels (tdvp_create, once per handle).
int qr_configure(Handle* h) {
  TDVP_CUDA(h, cudaFuncSetAttribute(k_qr_panel, cudaFuncAttributeMaxDynamicSharedMemorySize, SLAB_ROWS * NB * (int)sizeof(c128)));
  TDVP_CUDA(h, cudaFuncSetAttribute(k_qr_panel_cluster, cudaFuncAttributeMaxDynamicSharedMemorySize, CL_ROWS * NB * (int)sizeof(c128)));
  TDVP_CUDA(h, cudaFuncSetAttribute(k_qr_panel_cluster, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  h->qr_max_cluster = 0;
  for (int cs : {16, 8, 4, 2, 1}) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(cs);
    cfg.blockDim = dim3(32, CTY);
    cfg.dynamicSmemBytes = CL_ROWS * NB * sizeof(c128);
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int nclusters = 0;
    if (cudaOccupancyMaxActiveClusters(&nclusters, k_qr_panel_cluster, &cfg) == cudaSuccess && nclusters >= 1) { h->qr_max_cluster = cs; break; }
  }
  cudaGetLastError();
  if (h->num_sms > QR_MAX_SMS) { set_error(h, "qr: device has more SMs than the workspace bound"); return TDVP_ERR_UNSUPPORTED; }
  return 0;
}

// In-place economic QR of the row-major m x n matrix A (m >= n): on return Q (m x n, ld = ldq) and the upper
// triangle of A hold the factors.  Workspace comes from the handle's bump allocator.
int qr_factor(Handle* h, c128* A, int m, int n, int lda, c128* Q, int ldq) {
  if (m < n) { set_error(h, "qr_factor: needs m >= n"); return TDVP_ERR_SHAPE; }
  const int max_coop = h->num_sms;
  const int max_cluster = h->qr_max_cluster;
  const int qr_dbg = 0;
  const int np = (n + NB - 1) / NB;
  c128* Vall = (c128*)ws_alloc(h, sizeof(c128) * (size_t)m * lda);
  c128* Tall = (c128*)ws_alloc(h, sizeof(c128) * (size_t)np * NB * NB);
  c128* W = (c128*)ws_alloc(h, sizeof(c128) * (size_t)NB * n);
  c128* W2 = (c128*)ws_alloc(h, sizeof(c128) * (size_t)NB * n);
  double* tau = (double*)ws_alloc(h, sizeof(double) * 2 * (size_t)n);
  double* gpart = (double*)ws_alloc(h, sizeof(double) * 2 * (size_t)max_coop * 4 * NB);
  double* zpart = (double*)ws_alloc(h, sizeof(double) * 2 * (size_t)max_coop * NB * NB);
  // slabs of the panels taller than max_coop x SLAB_ROWS rows (the first panel is the tallest); G x rpc <= m + G rows
  c128* gslab = (m > max_coop * SLAB_ROWS) ? (c128*)ws_alloc(h, sizeof(c128) * (size_t)(m + max_coop) * NB) : nullptr;
  if (!Vall || !Tall || !W || !W2 || !tau || !gpart || !zpart || (m > max_coop * SLAB_ROWS && !gslab)) {
    set_error(h, "qr_factor: workspace");
    return TDVP_ERR_ARG;
  }
  TDVP_CUDA(h, cudaMemsetAsync(Vall, 0, sizeof(c128) * (size_t)m * lda, h->stream));
  const c128 one = {1.0, 0.0}, zero = {0.0, 0.0}, mone = {-1.0, 0.0};

  for (int pnl = 0; pnl < np; ++pnl) {
    const int j0 = pnl * NB;
    const int jb = (n - j0) < NB ? (n - j0) : NB;
    const int mp = m - j0;
    cudaError_t e;
    if (max_cluster >= 1 && mp <= max_cluster * CL_ROWS) {
      // one cluster owns the panel: pick the smallest power-of-two cluster that keeps <= 128 rows per CTA if possible
      int G = 1;
      constexpr int rows_target = 64;    // best of the sweep in scripts/debug/qr_timing.py
      while (G < max_cluster && (mp + G - 1) / G > rows_target) G *= 2;
      while ((mp + G - 1) / G > CL_ROWS) G *= 2;
      const int rpc = (mp + G - 1) / G;
      PanelArgs pa{A, lda, m, n, j0, jb, tau, Vall, Tall, gpart, zpart, rpc, nullptr, qr_dbg};
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(G);
      cfg.blockDim = dim3(32, CTY);
      cfg.dynamicSmemBytes = sizeof(c128) * (size_t)(rpc > 2 * NB ? rpc : 2 * NB) * NB;
      cfg.stream = h->stream;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeClusterDimension;
      at[0].val.clusterDim.x = G; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
      cfg.attrs = at; cfg.numAttrs = 1;
      { ProfScope _ps(h->stream, "qr.k_qr_panel_cluster"); e = cudaLaunchKernelEx(&cfg, k_qr_panel_cluster, pa); }
      count_launch();
      if (e != cudaSuccess) return cuda_fail(h, e, "cudaLaunchKernelEx(k_qr_panel_cluster)", __FILE__, __LINE__);
    } else {
      int rpc = SLAB_ROWS;
      int G = (mp + rpc - 1) / rpc;
      const bool global_slabs = G > max_coop;   // more slabs than SMs: one CTA per SM, slabs in global memory
      if (global_slabs) G = max_coop;
      if (G < 1) G = 1;
      rpc = (mp + G - 1) / G;  // spread rows evenly
      PanelArgs pa{A, lda, m, n, j0, jb, tau, Vall, Tall, gpart, zpart, rpc, global_slabs ? gslab : nullptr, qr_dbg};
      void* args[] = {&pa};
      const size_t smem = global_slabs ? 0 : sizeof(c128) * (size_t)(rpc > 2 * NB ? rpc : 2 * NB) * NB;
      { ProfScope _ps(h->stream, "qr.k_qr_panel"); e = cudaLaunchCooperativeKernel((void*)k_qr_panel, dim3(G), dim3(32, PTY), args, smem, h->stream); }
      count_launch();
      if (e != cudaSuccess) return cuda_fail(h, e, "cudaLaunchCooperativeKernel(k_qr_panel)", __FILE__, __LINE__);
    }
    const int nc = n - j0 - jb;
    if (nc > 0) {
      // C <- (I - V T^H V^H) C,  C = A[j0:, j0+jb:]
      c128* Vp = Vall + (long long)j0 * lda + j0;
      c128* C = A + (long long)j0 * lda + j0 + jb;
      c128* T = Tall + (size_t)pnl * NB * NB;
      TDVP_TRY(gemm(h, vhc_desc(jb, nc, mp, Vp, lda, C, lda, W, "qr.VhC")));     // W = V^H C
      TDVP_TRY(gemm(h, tagged(gemm_rowmajor(jb, nc, jb, T, NB, true, true, W, nc, false, W2, nc, one, zero), "qr.TW")));      // W2 = T^H W
      TDVP_TRY(gemm(h, tagged(gemm_rowmajor(mp, nc, jb, Vp, lda, false, false, W2, nc, false, C, lda, mone, one), "qr.VW"))); // C -= V W2
    }
  }
  // ---- form Q = H_1 ... H_k [I; 0]  (zungqr, blocked, backward) ----
  { ProfScope _ps(h->stream, "qr.k_set_identity"); k_set_identity<<<148 * 2, 256, 0, h->stream>>>(Q, m, n, ldq); }
  TDVP_TRY(lq(h, "k_set_identity"));
  for (int pnl = np - 1; pnl >= 0; --pnl) {
    const int j0 = pnl * NB;
    const int jb = (n - j0) < NB ? (n - j0) : NB;
    const int mp = m - j0;
    const int nc = n - j0;
    c128* Vp = Vall + (long long)j0 * lda + j0;
    c128* C = Q + (long long)j0 * ldq + j0;
    c128* T = Tall + (size_t)pnl * NB * NB;
    TDVP_TRY(gemm(h, vhc_desc(jb, nc, mp, Vp, lda, C, ldq, W, "ungqr.VhC")));      // W = V^H C
    TDVP_TRY(gemm(h, tagged(gemm_rowmajor(jb, nc, jb, T, NB, false, false, W, nc, false, W2, nc, one, zero), "ungqr.TW")));     // W2 = T W
    TDVP_TRY(gemm(h, tagged(gemm_rowmajor(mp, nc, jb, Vp, lda, false, false, W2, nc, false, C, ldq, mone, one), "ungqr.VW")));  // C -= V W2
  }
  return 0;
}

// Gauge shift of the centre tensor (see tdvp_qr_shift in include/tdvp_b200.h).
int qr_shift_exec(Handle* h, int gauge, int Dl, int d, int Dr, const c128* psi, c128* site, c128* sigma) {
  const long long N = (long long)Dl * d * Dr;
  const int m = (gauge == TDVP_GAUGE_A) ? Dl * d : Dr * d;
  const int n = (gauge == TDVP_GAUGE_A) ? Dr : Dl;
  if (m < n) { set_error(h, "qr_shift: matricisation has fewer rows than columns (bond dimension rule violated)"); return TDVP_ERR_SHAPE; }
  TDVP_TRY(ws_reserve(h, sizeof(c128) * (qr_ws_elems(m, n) + 2 * (size_t)N) + 4096));
  c128* Awork = (c128*)ws_alloc(h, sizeof(c128) * (size_t)N);
  if (!Awork) { set_error(h, "qr_shift: workspace"); return TDVP_ERR_ARG; }
  if (gauge == TDVP_GAUGE_A) {
    TDVP_CUDA(h, cudaMemcpyAsync(Awork, psi, sizeof(c128) * N, cudaMemcpyDeviceToDevice, h->stream));
    TDVP_TRY(qr_factor(h, Awork, m, n, n, site, n));                       // site(Dl,d,k=n) = Q
    { ProfScope _ps(h->stream, "qr.k_extract_r"); k_extract_r<<<64, 256, 0, h->stream>>>(Awork, n, n, n, sigma, n, 0); }   // sigma(k, Dr) = R
    TDVP_TRY(lq(h, "k_extract_r"));
  } else if (gauge == TDVP_GAUGE_B) {
    // QR of psi^T viewed as (Dr*d) x Dl;  B = Q reshaped (Dr,d,k) -> (k,d,Dr);  sigma = R^T (Dl, k)
    c128* Qt = (c128*)ws_alloc(h, sizeof(c128) * (size_t)N);
    if (!Qt) { set_error(h, "qr_shift: workspace"); return TDVP_ERR_ARG; }
    TDVP_TRY(permute_site(h, psi, Awork, Dl, d, Dr));                      // Awork[r,j,l] = psi[l,j,r]
    TDVP_TRY(qr_factor(h, Awork, m, n, n, Qt, n));
    TDVP_TRY(permute_site(h, Qt, site, Dr, d, n));                         // site[k,j,r] = Qt[r,j,k]
    { ProfScope _ps(h->stream, "qr.k_extract_r"); k_extract_r<<<64, 256, 0, h->stream>>>(Awork, n, n, n, sigma, n, 1); }   // sigma(Dl, k) = R^T
    TDVP_TRY(lq(h, "k_extract_r"));
  } else {
    set_error(h, "qr_shift: bad gauge");
    return TDVP_ERR_ARG;
  }
  return 0;
}

int absorb_exec(Handle* h, int gauge, int Dl, int d, int Dr, int k, const c128* sigma, const c128* site, c128* out) {
  TDVP_TRY(ws_reserve(h, 4096));
  if (gauge == TDVP_GAUGE_A) {
    // out(k, d*Dr) = sigma(k, Dl) . site(Dl, d*Dr)
    return gemm(h, tagged(gemm_rowmajor(k, d * Dr, Dl, sigma, Dl, false, false, site, (long long)d * Dr, false, out, (long long)d * Dr), "absorb"));
  } else if (gauge == TDVP_GAUGE_B) {
    // out(Dl*d, k) = site(Dl*d, Dr) . sigma(Dr, k)
    return gemm(h, tagged(gemm_rowmajor(Dl * d, k, Dr, site, Dr, false, false, sigma, k, false, out, k), "absorb"));
  }
  set_error(h, "absorb: bad gauge");
  return TDVP_ERR_ARG;
}

}  // namespace tdvp
