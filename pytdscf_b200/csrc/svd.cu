// Bond-matrix SVD, truncation and pseudo-inverse on the device.
//
// Replaces (reference file:line):
//   svd_exec + tdvp_svd_truncate   scipy.linalg.svd + cumulative-weight truncation in truncate_sigvec
//                                  (pytdscf/_site_cls.py:586-690)
//   tdvp_pinv                      np.linalg.pinv(X, rcond) in multiply_sigvec_pinv (pytdscf/_site_cls.py:709-754)
//
// Algorithm: one-sided (Hestenes) Jacobi on the columns of sigma, complex version: for a column pair (p, q) with
// gamma = g_p^H g_q = |gamma| e^{i phi} the pair (g_p, g_q e^{-i phi}) is rotated by the real Jacobi rotation that
// zeroes their inner product; V accumulates the same unitary, so sigma V = G at all times.  Pairs of one round of
// the round-robin tournament are independent and are spread over the CTAs of a cooperative grid (one grid sync per
// round).  One-sided Jacobi orthogonalises tiny columns to THEIR OWN scale (high relative accuracy), so U stays
// unitary down to the smallest non-zero singular value; exactly-zero columns are completed by a Householder QR of
// the padded matrix (the same LAPACK-style null-space completion the gauge shift uses).  That QR takes any row count, so
// tall rank-deficient inputs such as the (D_l D_r) x d matricisation of regularize_site with an empty physical level
// are completed too (above num_sms x 256 rows its panel slabs live in global memory).
#include <cooperative_groups.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "contract.cuh"

namespace cg = cooperative_groups;

namespace tdvp {

int qr_factor(Handle* h, c128* A, int m, int n, int lda, c128* Q, int ldq);
size_t qr_ws_elems(int m, int n);

namespace {

constexpr int JT = 256;

__device__ __forceinline__ void block_sum3(double& a, double& b, double& c, double& d_, double* sm) {
  // sums 4 doubles over the block; results broadcast to all threads
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  double v[4] = {a, b, c, d_};
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[i] += __shfl_xor_sync(0xffffffffu, v[i], o);
  __syncthreads();
  if (lane == 0) { sm[warp * 4 + 0] = v[0]; sm[warp * 4 + 1] = v[1]; sm[warp * 4 + 2] = v[2]; sm[warp * 4 + 3] = v[3]; }
  __syncthreads();
  double t[4] = {0, 0, 0, 0};
  for (int w = 0; w < nw; ++w) { t[0] += sm[w * 4]; t[1] += sm[w * 4 + 1]; t[2] += sm[w * 4 + 2]; t[3] += sm[w * 4 + 3]; }
  a = t[0]; b = t[1]; c = t[2]; d_ = t[3];
}

// Gt: n x m (row j = column j of sigma), Vt: n x n (row j = column j of V).  n may be odd (a bye is inserted).
// Columns whose norm falls below NEGLIGIBLE x (largest initial column norm) are numerical zeros: rotating them only
// reproduces rounding noise one ulp smaller each time (a rank-1 bond matrix of a padded Hartree product would rotate its
// noise columns until they underflow, ~20 sweeps); they are frozen, and svd_exec takes their left vectors from the
// orthonormal completion exactly like those of exact zeros.  LAPACK's gesdd resolves singular values only to
// eps x s_max, so nothing the reference can represent is lost (NEGLIGIBLE = 1e-20 << eps).
constexpr double NEGLIGIBLE = 1.0e-20;
constexpr double SIGNIFICANT = 8.0;     // see the rotation test in k_jacobi_svd

__global__ void __launch_bounds__(JT) k_jacobi_svd(c128* __restrict__ Gt, c128* __restrict__ Vt, int n, int m, int max_sweeps,
                                                    double tol, int* __restrict__ flags /* [0]: rotations in this sweep */,
                                                    unsigned long long* __restrict__ maxn2 /* zeroed: max |column|^2 as bits */) {
  __shared__ double sm[4 * (JT / 32)];
  cg::grid_group grid = cg::this_grid();
  const int ne = (n + 1) & ~1;           // players (even)
  const int npairs = ne / 2;
  for (int j = blockIdx.x; j < n; j += gridDim.x) {
    double a = 0.0, b = 0.0, c = 0.0, d = 0.0;
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
      const c128 x = Gt[(size_t)j * m + i];
      a += x.x * x.x + x.y * x.y;
    }
    block_sum3(a, b, c, d, sm);
    if (threadIdx.x == 0) atomicMax(maxn2, (unsigned long long)__double_as_longlong(a));   // non-negative doubles order like integers
    __syncthreads();
  }
  __threadfence();
  grid.sync();
  const double frozen2 = NEGLIGIBLE * NEGLIGIBLE * __longlong_as_double((long long)*((volatile unsigned long long*)maxn2));
  for (int sweep = 0; sweep < max_sweeps; ++sweep) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      flags[(sweep + 1) % 3] = 0;   // reset the counter of the NEXT sweep (3 slots: no reader of slot sweep-1 is disturbed)
      reinterpret_cast<unsigned long long*>(flags + 8)[(sweep + 1) % 3] = 0ull;    // ... and its largest |cos| (as bits)
    }
    for (int r = 0; r < ne - 1; ++r) {
      for (int t = blockIdx.x; t < npairs; t += gridDim.x) {
        int p, q;
        if (t == 0) { p = ne - 1; q = r; }
        else { p = (r + t) % (ne - 1); q = (r - t + (ne - 1)) % (ne - 1); }
        if (p >= n || q >= n) continue;   // bye
        if (p > q) { const int x = p; p = q; q = x; }
        c128* gp = Gt + (size_t)p * m;
        c128* gq = Gt + (size_t)q * m;
        double al = 0.0, be = 0.0, gr = 0.0, gi = 0.0;
        for (int i = threadIdx.x; i < m; i += blockDim.x) {
          const c128 x = gp[i], y = gq[i];
          al += x.x * x.x + x.y * x.y;
          be += y.x * y.x + y.y * y.y;
          gr += x.x * y.x + x.y * y.y;   // conj(x) * y
          gi += x.x * y.y - x.y * y.x;
        }
        block_sum3(al, be, gr, gi, sm);
        const double ga = hypot(gr, gi);
        const double lim = tol * sqrt(al) * sqrt(be);
        if (al > frozen2 && be > frozen2 && ga > lim) {
          // every pair above the threshold is rotated, but only rotations clearly above the rounding level of the inner
          // product (SIGNIFICANT x threshold) keep the sweeps going: at the threshold itself rounding alone re-creates
          // inner products of that size, and a 512 x 512 bond matrix was seen to flip such pairs for 40 sweeps
          if (threadIdx.x == 0 && ga > SIGNIFICANT * lim) {
            atomicAdd(&flags[sweep % 3], 1);
            atomicMax(reinterpret_cast<unsigned long long*>(flags + 8) + sweep % 3,
                      (unsigned long long)__double_as_longlong(ga / (sqrt(al) * sqrt(be))));
          }
          const double pr = gr / ga, pi = gi / ga;          // e^{i phi}
          const double zeta = (be - al) / (2.0 * ga);
          const double tt = (zeta >= 0.0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
          const double c = 1.0 / sqrt(1.0 + tt * tt), s = c * tt;
          for (int i = threadIdx.x; i < m; i += blockDim.x) {
            const c128 x = gp[i], y = gq[i];
            const c128 yt = {y.x * pr + y.y * pi, y.y * pr - y.x * pi};   // y * e^{-i phi}
            gp[i] = {c * x.x - s * yt.x, c * x.y - s * yt.y};
            gq[i] = {s * x.x + c * yt.x, s * x.y + c * yt.y};
          }
          c128* vp = Vt + (size_t)p * n;
          c128* vq = Vt + (size_t)q * n;
          for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const c128 x = vp[i], y = vq[i];
            const c128 yt = {y.x * pr + y.y * pi, y.y * pr - y.x * pi};
            vp[i] = {c * x.x - s * yt.x, c * x.y - s * yt.y};
            vq[i] = {s * x.x + c * yt.x, s * x.y + c * yt.y};
          }
        }
        __syncthreads();
      }
      __threadfence();
      grid.sync();
    }
    const int nrot = *((volatile int*)&flags[sweep % 3]);
    if (nrot == 0) {
      if (blockIdx.x == 0 && threadIdx.x == 0) flags[3] = 1;   // converged: a full sweep without a significant rotation
      break;
    }
    if (sweep == max_sweeps - 1 && blockIdx.x == 0 && threadIdx.x == 0) {
      // out of sweeps: report how far from orthogonal the columns still were in the last one (svd_exec decides)
      reinterpret_cast<unsigned long long*>(flags + 8)[3] = *((volatile unsigned long long*)(reinterpret_cast<unsigned long long*>(flags + 8) + sweep % 3));
    }
  }
}

// ---- blocked variant: the columns are grouped into blocks of B; one CTA owns a PAIR of blocks for a tournament round,
// holds their 2B columns (each of length m) in shared memory and rotates every column pair that meets there -- all B*B cross
// pairs, plus (in the first round of a sweep) the pairs inside each block -- with one warp per pair and only CTA-level
// barriers in between.  The unitary accumulated for the 2B columns is applied to the matching 2B columns of V once per
// task.  A sweep therefore costs n/B - 1 grid-wide barriers instead of n - 1, and a matrix of up to 2B columns needs none
// at all (r1: 511 grid barriers per sweep at n = 512 made the plain kernel latency-bound at 35 ms).
constexpr int BJ_THREADS = 256;
constexpr int BJ_WARPS = BJ_THREADS / 32;
constexpr int BJ_SMEM_COLS_BYTES = 160 * 1024;     // budget for the 2B resident columns

__device__ __forceinline__ int bj_rotate_pair(c128* __restrict__ xp, c128* __restrict__ xq, int m, c128* __restrict__ wp,
                                              c128* __restrict__ wq, int w2, double tol, double frozen2, int lane) {
  double al = 0.0, be = 0.0, gr = 0.0, gi = 0.0;
  for (int i = lane; i < m; i += 32) {
    const c128 x = xp[i], y = xq[i];
    al += x.x * x.x + x.y * x.y;
    be += y.x * y.x + y.y * y.y;
    gr += x.x * y.x + x.y * y.y;   // conj(x) * y
    gi += x.x * y.y - x.y * y.x;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    al += __shfl_xor_sync(0xffffffffu, al, o);
    be += __shfl_xor_sync(0xffffffffu, be, o);
    gr += __shfl_xor_sync(0xffffffffu, gr, o);
    gi += __shfl_xor_sync(0xffffffffu, gi, o);
  }
  const double ga = hypot(gr, gi);
  const double lim = tol * sqrt(al) * sqrt(be);
  if (!(al > frozen2 && be > frozen2 && ga > lim)) return 0;
  const int significant = ga > SIGNIFICANT * lim ? 0x10000 : 0;    // high half: rotations that keep the sweeps going
  const double pr = gr / ga, pi = gi / ga;          // e^{i phi}
  const double zeta = (be - al) / (2.0 * ga);
  const double tt = (zeta >= 0.0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
  const double c = 1.0 / sqrt(1.0 + tt * tt), s = c * tt;
  for (int i = lane; i < m; i += 32) {
    const c128 x = xp[i], y = xq[i];
    const c128 yt = {y.x * pr + y.y * pi, y.y * pr - y.x * pi};   // y * e^{-i phi}
    xp[i] = {c * x.x - s * yt.x, c * x.y - s * yt.y};
    xq[i] = {s * x.x + c * yt.x, s * x.y + c * yt.y};
  }
  for (int i = lane; i < w2; i += 32) {
    const c128 x = wp[i], y = wq[i];
    const c128 yt = {y.x * pr + y.y * pi, y.y * pr - y.x * pi};
    wp[i] = {c * x.x - s * yt.x, c * x.y - s * yt.y};
    wq[i] = {s * x.x + c * yt.x, s * x.y + c * yt.y};
  }
  return 1 + significant;
}

__global__ void __launch_bounds__(BJ_THREADS, 1)
    k_jacobi_svd_blocked(c128* __restrict__ Gt, c128* __restrict__ Vt, int n, int m, int B, int max_sweeps, double tol,
                         int* __restrict__ flags, unsigned long long* __restrict__ maxn2) {
  extern __shared__ __align__(16) unsigned char bj_smem[];
  c128* X = reinterpret_cast<c128*>(bj_smem);              // [2B][m]: rows 0..B-1 = block I, B..2B-1 = block J
  c128* Wt = X + (size_t)2 * B * m;                        // [2B][2B]: accumulated transformation of the 2B rows
  __shared__ double sm[4 * (BJ_THREADS / 32)];
  __shared__ int s_rot;
  cg::grid_group grid = cg::this_grid();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int W2 = 2 * B;
  const int nblk = (n + B - 1) / B;
  const int ne = (nblk + 1) & ~1;                          // players (blocks), even
  const int ntask = ne / 2;
  // largest initial column norm (see NEGLIGIBLE)
  for (int j = blockIdx.x; j < n; j += gridDim.x) {
    double a = 0.0, b2 = 0.0, c2 = 0.0, d2 = 0.0;
    for (int i = tid; i < m; i += blockDim.x) {
      const c128 x = Gt[(size_t)j * m + i];
      a += x.x * x.x + x.y * x.y;
    }
    block_sum3(a, b2, c2, d2, sm);
    if (tid == 0) atomicMax(maxn2, (unsigned long long)__double_as_longlong(a));
    __syncthreads();
  }
  __threadfence();
  grid.sync();
  const double frozen2 = NEGLIGIBLE * NEGLIGIBLE * __longlong_as_double((long long)*((volatile unsigned long long*)maxn2));

  for (int sweep = 0; sweep < max_sweeps; ++sweep) {
    if (blockIdx.x == 0 && tid == 0) flags[(sweep + 1) % 3] = 0;
    const int nrounds = ne > 1 ? ne - 1 : 1;
    for (int r = 0; r < nrounds; ++r) {
      for (int t = blockIdx.x; t < ntask; t += gridDim.x) {
        int bI, bJ;
        if (ne == 1) { bI = 0; bJ = 1; }
        else if (t == 0) { bI = ne - 1; bJ = r; }
        else { bI = (r + t) % (ne - 1); bJ = (r - t + (ne - 1)) % (ne - 1); }
        if (bI > bJ) { const int x = bI; bI = bJ; bJ = x; }
        const bool haveJ = bJ < nblk;
        if (bI >= nblk) continue;                            // both byes (cannot happen for bI < bJ, kept for safety)
        if (!haveJ && r != 0) continue;                      // bye: only the in-block pairs of round 0 remain to be done
        // ---- load the 2B columns (rows of Gt), zero rows for columns beyond n / the bye block ----
        for (int row = 0; row < W2; ++row) {
          const int gcol = (row < B ? bI * B + row : bJ * B + (row - B));
          const bool ok = gcol < n && (row < B || haveJ);
          const c128* src = Gt + (size_t)gcol * m;
          for (int i = tid; i < m; i += BJ_THREADS) X[(size_t)row * m + i] = ok ? src[i] : c128{0.0, 0.0};
        }
        for (int e = tid; e < W2 * W2; e += BJ_THREADS) Wt[e] = {(e / W2 == e % W2) ? 1.0 : 0.0, 0.0};
        if (tid == 0) s_rot = 0;
        __syncthreads();
        int my_rot = 0;
        // ---- pairs inside the two blocks (first round of the sweep only): round-robin over B players ----
        if (r == 0 && B > 1) {
          for (int rr = 0; rr < B - 1; ++rr) {
            for (int pr_ = warp; pr_ < B; pr_ += BJ_WARPS) {     // B/2 pairs per block, two blocks
              const int blk = pr_ / (B / 2), tt_ = pr_ % (B / 2);
              int p, q;
              if (tt_ == 0) { p = B - 1; q = rr; }
              else { p = (rr + tt_) % (B - 1); q = (rr - tt_ + (B - 1)) % (B - 1); }
              if (p > q) { const int x = p; p = q; q = x; }
              p += blk * B; q += blk * B;
              my_rot += bj_rotate_pair(X + (size_t)p * m, X + (size_t)q * m, m, Wt + p * W2, Wt + q * W2, W2, tol, frozen2, lane);
            }
            __syncthreads();
          }
        }
        // ---- cross pairs: B rounds of B disjoint pairs (i, B + (i + rr) mod B) ----
        if (haveJ) {
          for (int rr = 0; rr < B; ++rr) {
            for (int i = warp; i < B; i += BJ_WARPS) {
              const int p = i, q = B + (i + rr) % B;
              my_rot += bj_rotate_pair(X + (size_t)p * m, X + (size_t)q * m, m, Wt + p * W2, Wt + q * W2, W2, tol, frozen2, lane);
            }
            __syncthreads();
          }
        }
        if (lane == 0 && my_rot) atomicAdd(&s_rot, my_rot);
        __syncthreads();
        const int rot = s_rot;                             // low half: rotations applied, high half: significant ones
        if (rot > 0) {
          if (tid == 0 && (rot >> 16) > 0) atomicAdd(&flags[sweep % 3], rot >> 16);
          // ---- write the columns back and apply the accumulated transformation to the same columns of V ----
          for (int row = 0; row < W2; ++row) {
            const int gcol = (row < B ? bI * B + row : bJ * B + (row - B));
            if (!(gcol < n && (row < B || haveJ))) continue;
            c128* dst = Gt + (size_t)gcol * m;
            for (int i = tid; i < m; i += BJ_THREADS) dst[i] = X[(size_t)row * m + i];
          }
          for (int col = tid; col < n; col += BJ_THREADS) {
            c128 vold[32], vnew;
#pragma unroll
            for (int k = 0; k < 32; ++k) {
              if (k < W2) {
                const int gcol = (k < B ? bI * B + k : bJ * B + (k - B));
                vold[k] = (gcol < n && (k < B || haveJ)) ? Vt[(size_t)gcol * n + col] : c128{0.0, 0.0};
              }
            }
            for (int j = 0; j < W2; ++j) {
              const int gcol = (j < B ? bI * B + j : bJ * B + (j - B));
              if (!(gcol < n && (j < B || haveJ))) continue;
              vnew = {0.0, 0.0};
#pragma unroll
              for (int k = 0; k < 32; ++k) {
                if (k < W2) {
                  const c128 w = Wt[j * W2 + k];
                  vnew.x += w.x * vold[k].x - w.y * vold[k].y;
                  vnew.y += w.x * vold[k].y + w.y * vold[k].x;
                }
              }
              Vt[(size_t)gcol * n + col] = vnew;
            }
          }
        }
        __syncthreads();
      }
      if (ne > 2) { __threadfence(); grid.sync(); }
    }
    if (ne <= 2) { __threadfence(); __syncthreads(); }
    const int nrot = *((volatile int*)&flags[sweep % 3]);
    if (nrot == 0) {
      if (blockIdx.x == 0 && tid == 0) flags[3] = 1;
      break;
    }
    if (ne <= 2) __syncthreads();
  }
}

// norms[j] = |Gt[j, :]|
__global__ void k_row_norms(const c128* __restrict__ Gt, int n, int m, double* __restrict__ norms) {
  __shared__ double sm[4 * (JT / 32)];
  for (int j = blockIdx.x; j < n; j += gridDim.x) {
    double a = 0.0, b = 0.0, c = 0.0, d = 0.0;
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
      const c128 x = Gt[(size_t)j * m + i];
      a += x.x * x.x + x.y * x.y;
    }
    block_sum3(a, b, c, d, sm);
    if (threadIdx.x == 0) norms[j] = sqrt(a);
    __syncthreads();
  }
}

// U[i, jj] = Gt[perm[jj], i] / s[jj] (zero column when s == 0); Vh[jj, i] = conj(Vt[perm[jj], i])
__global__ void k_assemble_uv(const c128* __restrict__ Gt, const c128* __restrict__ Vt, const int* __restrict__ perm,
                              const double* __restrict__ s, int n, int m, c128* __restrict__ U, int ldu,
                              c128* __restrict__ Vh, int ldv) {
  const long long totU = (long long)m * n, totV = (long long)n * n;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < totU + totV; e += (long long)gridDim.x * blockDim.x) {
    if (e < totU) {
      const int i = (int)(e / n), jj = (int)(e % n);
      const double sv = s[jj];
      c128 g = Gt[(size_t)perm[jj] * m + i];
      if (sv > 0.0) { g.x /= sv; g.y /= sv; } else { g.x = 0.0; g.y = 0.0; }
      U[(size_t)i * ldu + jj] = g;
    } else {
      const long long f = e - totU;
      const int jj = (int)(f / n), i = (int)(f % n);
      const c128 v = Vt[(size_t)perm[jj] * n + i];
      Vh[(size_t)jj * ldv + i] = {v.x, -v.y};
    }
  }
}

// copy columns [c0, c1) of src (ld lds) into the same columns of dst (ld ldd), m rows
__global__ void k_copy_cols(const c128* __restrict__ src, int lds, c128* __restrict__ dst, int ldd, int m, int c0, int c1) {
  const int w = c1 - c0;
  const long long tot = (long long)m * w;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(e / w), j = c0 + (int)(e % w);
    dst[(size_t)i * ldd + j] = src[(size_t)i * lds + j];
  }
}

// rows[j, :] *= f[j]
__global__ void k_scale_rows(c128* __restrict__ A, int rows, int cols, int ld, const double* __restrict__ f) {
  const long long tot = (long long)rows * cols;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(e / cols), j = (int)(e % cols);
    c128& v = A[(size_t)i * ld + j];
    v.x *= f[i];
    v.y *= f[i];
  }
}

__global__ void k_identity(c128* __restrict__ A, int n) {
  const long long tot = (long long)n * n;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x)
    A[e] = {(e / n == e % n) ? 1.0 : 0.0, 0.0};
}

__global__ void k_diag_matrix(c128* __restrict__ S, int k, const double* __restrict__ vals) {
  const long long tot = (long long)k * k;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(e / k), j = (int)(e % k);
    S[e] = {i == j ? vals[i] : 0.0, 0.0};
  }
}

// max |off-diagonal| and max |diagonal| of an n x n matrix (one CTA; n <= a few thousand)
__global__ void k_diag_probe(const c128* __restrict__ X, int n, double* __restrict__ out2) {
  __shared__ double s_off[32], s_dia[32];
  double off = 0.0, dia = 0.0;
  const long long tot = (long long)n * n;
  for (long long e = threadIdx.x; e < tot; e += blockDim.x) {
    const c128 v = X[e];
    const double a = fmax(fabs(v.x), fabs(v.y));
    if (e / n == e % n) dia = fmax(dia, hypot(v.x, v.y)); else off = fmax(off, a);
  }
  for (int o = 16; o > 0; o >>= 1) {
    off = fmax(off, __shfl_xor_sync(0xffffffffu, off, o));
    dia = fmax(dia, __shfl_xor_sync(0xffffffffu, dia, o));
  }
  if ((threadIdx.x & 31) == 0) { s_off[threadIdx.x >> 5] = off; s_dia[threadIdx.x >> 5] = dia; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { off = fmax(off, s_off[w]); dia = fmax(dia, s_dia[w]); }
    out2[0] = off; out2[1] = dia;
  }
}

// pseudo-inverse of a diagonal matrix: 1/d_i where |d_i| > rcond * max|d|, else 0
__global__ void k_pinv_diag(const c128* __restrict__ X, int n, double cut, c128* __restrict__ out) {
  const long long tot = (long long)n * n;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x) {
    c128 r = {0.0, 0.0};
    if (e / n == e % n) {
      const c128 v = X[e];
      const double a2 = v.x * v.x + v.y * v.y;
      if (sqrt(a2) > cut) r = {v.x / a2, -v.y / a2};
    }
    out[e] = r;
  }
}

int ls(Handle* h, const char* what) {
  count_launch();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(h, e, what, __FILE__, __LINE__);
  return 0;
}

// Orthonormal completion of the last (n - r) columns of the m x n matrix U whose first r columns are orthonormal:
// Householder QR of [U_r | 0] gives Q whose trailing columns span the orthogonal complement.
int complete_columns(Handle* h, c128* U, int m, int n, int ldu, int r) {
  if (r >= n) return 0;
  c128* W = (c128*)ws_alloc(h, sizeof(c128) * (size_t)m * n);
  c128* Q = (c128*)ws_alloc(h, sizeof(c128) * (size_t)m * n);
  if (!W || !Q) { set_error(h, "svd: workspace (completion)"); return TDVP_ERR_ARG; }
  TDVP_CUDA(h, cudaMemsetAsync(W, 0, sizeof(c128) * (size_t)m * n, h->stream));
  if (r > 0) {
    k_copy_cols<<<148, 256, 0, h->stream>>>(U, ldu, W, n, m, 0, r);
    TDVP_TRY(ls(h, "k_copy_cols"));
  }
  TDVP_TRY(qr_factor(h, W, m, n, n, Q, n));
  k_copy_cols<<<148, 256, 0, h->stream>>>(Q, n, U, ldu, m, r, n);
  return ls(h, "k_copy_cols");
}

}  // namespace

int svd_configure(Handle* h) {
  int per = 0;
  TDVP_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_jacobi_svd, JT, 0));
  h->svd_max_blocks = h->num_sms * (per > 4 ? 4 : (per < 1 ? 1 : per));
  const int smem = BJ_SMEM_COLS_BYTES + 4 * 16 * 16 * (int)sizeof(c128);
  TDVP_CUDA(h, cudaFuncSetAttribute(k_jacobi_svd_blocked, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  per = 0;
  TDVP_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_jacobi_svd_blocked, BJ_THREADS, smem));
  h->svd_blocked_max_blocks = h->num_sms * (per < 1 ? 0 : 1);
  return 0;
}

// Thin SVD sigma(m x n, row-major, m >= n) = U(m x n) diag(s) Vh(n x n); s descending, copied to host_s.
size_t svd_ws_bytes(int m, int n) {
  return sizeof(c128) * ((size_t)n * m + (size_t)n * n + 2 * (size_t)m * n + qr_ws_elems(m, n)) +
         sizeof(double) * 8 * (size_t)n + 8192;   // incl. the n doubles tdvp_svd_truncate / tdvp_pinv add afterwards
}

// `reserve` false: the caller has reserved svd_ws_bytes(m, n) beyond what it already took from the bump allocator.
int svd_exec(Handle* h, int m, int n, const c128* sigma, c128* U, c128* Vh, double* host_s, bool reserve = true) {
  if (m < n) { set_error(h, "svd: needs m >= n"); return TDVP_ERR_SHAPE; }
  if (reserve) TDVP_TRY(ws_reserve(h, svd_ws_bytes(m, n)));
  c128* Gt = (c128*)ws_alloc(h, sizeof(c128) * (size_t)n * m);
  c128* Vt = (c128*)ws_alloc(h, sizeof(c128) * (size_t)n * n);
  double* norms = (double*)ws_alloc(h, sizeof(double) * n);
  double* svals = (double*)ws_alloc(h, sizeof(double) * n);
  int* perm = (int*)ws_alloc(h, sizeof(int) * n);
  int* flags = (int*)ws_alloc(h, sizeof(int) * 16);  // [0..2] rotation counters, [3] converged, [4..5] max |column|^2, [8..15] max |cos| per sweep slot + final
  if (!Gt || !Vt || !norms || !svals || !perm || !flags) { set_error(h, "svd: workspace"); return TDVP_ERR_ARG; }
  cudaStream_t st = h->stream;
  TDVP_TRY(permute_site(h, sigma, Gt, m, 1, n));   // Gt[j, i] = sigma[i, j]
  { ProfScope _ps(st, "svd.k_identity"); k_identity<<<148, 256, 0, st>>>(Vt, n); }
  TDVP_TRY(ls(h, "k_identity"));
  TDVP_CUDA(h, cudaMemsetAsync(flags, 0, sizeof(int) * 16, st));
  unsigned long long* maxn2 = reinterpret_cast<unsigned long long*>(flags + 4);
  {
    int max_sweeps = 60;
    // LAPACK zgesvj's threshold: sqrt(m) * eps -- the rounding level of an m-term inner product.  A fixed 1e-15 sits
    // below that noise for m in the hundreds and would keep rotating (and never report convergence).
    double tol = std::sqrt((double)m) * 2.220446049250313e-16;
    cudaError_t e;
    // columns per block of the blocked kernel: as many as fit the shared-memory budget (two blocks resident), at most 16,
    // and no more than half of the matrix (two blocks then hold everything and the whole SVD runs without a grid barrier)
    int Bmax = 0;
    for (int b = 16; b >= 2; b >>= 1)
      if ((size_t)2 * b * m * sizeof(c128) <= (size_t)BJ_SMEM_COLS_BYTES) { Bmax = b; break; }
    int B = 2;
    while (B < Bmax && 2 * B < n) B <<= 1;
    // Measured (profiles/r2_svd_qr_latency.jsonl): with several block pairs per round the blocked kernel is SLOWER than
    // the plain one (48 vs 35 ms at 512 x 512: 8 warps per resident block pair cannot hide the ~2 us FP64 sqrt / division
    // chain of each rotation, and only n / 2B CTAs are busy), so it is used where it needs no grid barrier at all:
    // matrices whose columns fit one block pair (n <= 2B <= 32 -- the bond matrices of the small-D regime).
    if (Bmax >= 2 && 2 * B >= n && h->svd_blocked_max_blocks >= 1) {
      const int nblk = (n + B - 1) / B;
      const int ntask = ((nblk + 1) & ~1) / 2;
      int grid = ntask < h->svd_blocked_max_blocks ? ntask : h->svd_blocked_max_blocks;
      if (grid < 1) grid = 1;
      const size_t smem = sizeof(c128) * ((size_t)2 * B * m + (size_t)4 * B * B);
      void* args[] = {&Gt, &Vt, &n, &m, &B, &max_sweeps, &tol, &flags, &maxn2};
      { ProfScope _ps(st, "svd.k_jacobi_svd_blocked"); e = cudaLaunchCooperativeKernel((void*)k_jacobi_svd_blocked, dim3(grid), dim3(BJ_THREADS), args, smem, st); }
      count_launch();
      if (e != cudaSuccess) return cuda_fail(h, e, "cudaLaunchCooperativeKernel(k_jacobi_svd_blocked)", __FILE__, __LINE__);
    } else {
      // very long columns (tall-skinny inputs such as the (D_l D_r) x d matricisation of regularize_site): one CTA per
      // column pair, streaming from HBM
      const int max_blocks = h->svd_max_blocks;
      int grid = (n + 1) / 2;
      if (grid > max_blocks) grid = max_blocks;
      if (grid < 1) grid = 1;
      void* args[] = {&Gt, &Vt, &n, &m, &max_sweeps, &tol, &flags, &maxn2};
      { ProfScope _ps(st, "svd.k_jacobi_svd"); e = cudaLaunchCooperativeKernel((void*)k_jacobi_svd, dim3(grid), dim3(JT), args, 0, st); }
      count_launch();
      if (e != cudaSuccess) return cuda_fail(h, e, "cudaLaunchCooperativeKernel(k_jacobi_svd)", __FILE__, __LINE__);
    }
  }
  k_row_norms<<<148, JT, 0, st>>>(Gt, n, m, norms);
  TDVP_TRY(ls(h, "k_row_norms"));
  std::vector<double> hn(n);
  int conv = 0;
  double last_cos = 0.0;
  TDVP_CUDA(h, cudaMemcpyAsync(hn.data(), norms, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
  TDVP_CUDA(h, cudaMemcpyAsync(&conv, flags + 3, sizeof(int), cudaMemcpyDeviceToHost, st));
  TDVP_CUDA(h, cudaMemcpyAsync(&last_cos, flags + 14, sizeof(double), cudaMemcpyDeviceToHost, st));
  TDVP_CUDA(h, cudaStreamSynchronize(st));
  // Out of sweeps: accept when the columns were orthogonal to 1e-10 in the last sweep (rounding-level rotations that never
  // die out completely), fail otherwise -- an unconverged factorisation must not reach truncate_sigvec / pinv / Kraus.
  if (!conv && !(last_cos > 0.0 && last_cos < 1.0e-10)) {
    char msg[160];
    snprintf(msg, sizeof(msg), "svd: one-sided Jacobi did not converge in 60 sweeps (largest |cos| between columns in the last sweep: %.3e)", last_cos);
    set_error(h, msg);
    return TDVP_ERR_NOT_CONVERGED;
  }
  // ordering of the (already computed) singular values is index bookkeeping: descending, stable
  std::vector<int> hp(n);
  for (int i = 0; i < n; ++i) hp[i] = i;
  std::stable_sort(hp.begin(), hp.end(), [&](int a, int b) { return hn[a] > hn[b]; });
  std::vector<double> hs(n);
  int r = 0;
  // Columns the kernel froze as numerical zeros (norm < NEGLIGIBLE x largest initial column norm <= NEGLIGIBLE x s_max)
  // can never pass this test, so every un-orthogonalised column gets its left vector from the orthonormal completion,
  // like the columns of exactly zero singular values.  The computed value is still reported.
  for (int i = 0; i < n; ++i) { hs[i] = hn[hp[i]]; if (hs[i] > 0.0 && hs[i] > 4.0 * NEGLIGIBLE * hs[0]) r = i + 1; }
  TDVP_CUDA(h, cudaMemcpyAsync(perm, hp.data(), sizeof(int) * n, cudaMemcpyHostToDevice, st));
  TDVP_CUDA(h, cudaMemcpyAsync(svals, hs.data(), sizeof(double) * n, cudaMemcpyHostToDevice, st));
  k_assemble_uv<<<148 * 2, 256, 0, st>>>(Gt, Vt, perm, svals, n, m, U, n, Vh, n);
  TDVP_TRY(ls(h, "k_assemble_uv"));
  TDVP_CUDA(h, cudaStreamSynchronize(st));   // hp / hs are host temporaries
  if (r < n) TDVP_TRY(complete_columns(h, U, m, n, n, r));
  for (int i = 0; i < n; ++i) host_s[i] = hs[i];
  return 0;
}

}  // namespace tdvp

using namespace tdvp;

extern "C" {

int tdvp_svd_truncate(tdvp_handle_t hh, int m, int n, const tdvp_c128* sigma, double p, int keepdim, int regularize,
                      tdvp_c128* U, tdvp_c128* S, tdvp_c128* Vh, int* rank) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h) return TDVP_ERR_ARG;
  h->err.clear();
  if (!sigma || !U || !S || !Vh || !rank || m <= 0 || n <= 0 || m != n) {
    set_error(h, "svd_truncate: bad argument (the bond matrix must be square)");
    return TDVP_ERR_ARG;
  }
  std::vector<double> s(n);
  TDVP_TRY(svd_exec(h, m, n, (const c128*)sigma, (c128*)U, (c128*)Vh, s.data()));
  // cumulative singular-VALUE weight (not squared), first index with contribution >= 1 - p  (_site_cls.py:629-634)
  std::vector<double> cs(n);
  double acc = 0.0;
  for (int i = 0; i < n; ++i) { acc += s[i]; cs[i] = acc; }
  int idx = n;
  for (int i = 0; i < n; ++i) if (cs[i] / cs[n - 1] >= 1.0 - p) { idx = i + 1; break; }
  std::vector<double> thin(s.begin(), s.begin() + idx);
  const double sqrt_epsrho = 1.0e-4;   // SQRT_EPSRHO, _site_cls.py:22
  if (regularize && !(m == 1 && n == 1))
    for (double& v : thin) if (!(v > sqrt_epsrho)) v = v + sqrt_epsrho * std::exp(-v / sqrt_epsrho);
  double nrm = 0.0;
  for (double v : thin) nrm += v * v;
  nrm = std::sqrt(nrm);
  const int k = keepdim ? n : idx;
  std::vector<double> diag(k, 0.0);
  for (int i = 0; i < idx; ++i) diag[i] = thin[i] / nrm;
  double* dvals = (double*)ws_alloc(h, sizeof(double) * k);
  if (!dvals) { set_error(h, "svd_truncate: workspace"); return TDVP_ERR_ARG; }
  TDVP_CUDA(h, cudaMemcpyAsync(dvals, diag.data(), sizeof(double) * k, cudaMemcpyHostToDevice, h->stream));
  k_diag_matrix<<<148, 256, 0, h->stream>>>((c128*)S, k, dvals);
  count_launch();
  TDVP_CUDA(h, cudaStreamSynchronize(h->stream));
  // without keepdim the caller uses the leading idx columns of U (ld n) and rows of Vh
  *rank = idx;
  return 0;
}

int tdvp_svd(tdvp_handle_t hh, int m, int n, const tdvp_c128* A, tdvp_c128* U, double* s_host, tdvp_c128* Vh) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h) return TDVP_ERR_ARG;
  h->err.clear();
  if (!A || !U || !s_host || !Vh || m <= 0 || n <= 0 || m < n) { set_error(h, "svd: bad argument (needs m >= n)"); return TDVP_ERR_ARG; }
  return svd_exec(h, m, n, (const c128*)A, (c128*)U, (c128*)Vh, s_host);
}

int tdvp_pinv(tdvp_handle_t hh, int m, int n, const tdvp_c128* X, double rcond, tdvp_c128* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h) return TDVP_ERR_ARG;
  h->err.clear();
  if (!X || !out || m <= 0 || n <= 0 || m != n) { set_error(h, "pinv: bad argument (square matrices only)"); return TDVP_ERR_ARG; }
  // Bond matrices handed over by the site-parallel scheme are diagonal (the S of truncate_sigvec) in every step but
  // the first: their pseudo-inverse needs no SVD.
  {
    k_diag_probe<<<1, 1024, 0, h->stream>>>((const c128*)X, n, h->d_scal + 4000);
    TDVP_TRY(ls(h, "k_diag_probe"));
    TDVP_CUDA(h, cudaMemcpyAsync(h->h_scal + 4000, h->d_scal + 4000, 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    TDVP_CUDA(h, cudaStreamSynchronize(h->stream));
    if (h->h_scal[4000] == 0.0) {
      k_pinv_diag<<<148, 256, 0, h->stream>>>((const c128*)X, n, rcond * h->h_scal[4001], (c128*)out);
      return ls(h, "k_pinv_diag");
    }
  }
  // General (non-diagonal) input: only the very first step of a site-parallel run gets here.  U / Vh live in the handle's
  // workspace, reserved together with what the SVD itself needs (no allocation on this path).
  TDVP_TRY(ws_reserve(h, svd_ws_bytes(m, n) + 2 * align256(sizeof(c128) * (size_t)m * n) + 4096));
  c128* U = (c128*)ws_alloc(h, sizeof(c128) * (size_t)m * n);
  c128* Vh = (c128*)ws_alloc(h, sizeof(c128) * (size_t)n * n);
  if (!U || !Vh) { set_error(h, "pinv: workspace"); return TDVP_ERR_ARG; }
  std::vector<double> s(n);
  TDVP_TRY(svd_exec(h, m, n, (const c128*)X, U, Vh, s.data(), false));
  std::vector<double> inv(n);
  const double cut = rcond * s[0];
  for (int i = 0; i < n; ++i) inv[i] = (s[i] > cut) ? 1.0 / s[i] : 0.0;
  double* dinv = (double*)ws_alloc(h, sizeof(double) * n);
  if (!dinv) { set_error(h, "pinv: workspace"); return TDVP_ERR_ARG; }
  TDVP_CUDA(h, cudaMemcpyAsync(dinv, inv.data(), sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
  k_scale_rows<<<148, 256, 0, h->stream>>>(Vh, n, n, n, dinv);
  TDVP_TRY(ls(h, "k_scale_rows"));
  // out(n x m) = Vh^H (n x k) . U^H (k x m)
  GemmDesc g = gemm_rowmajor(n, m, n, Vh, n, true, true, U, n, true, (c128*)out, m);
  g.b_conj = 1;
  g.tag = "pinv";
  TDVP_TRY(gemm(h, g, "zgemm(pinv)"));
  TDVP_CUDA(h, cudaStreamSynchronize(h->stream));   // `inv` is a host temporary of the copy above
  return 0;
}

}  // extern "C"
