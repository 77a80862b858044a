// Short-iterative Lanczos / Arnoldi exponential with the reference's exact control flow, Krylov
// vectors resident in HBM, fused HBM-bound vector kernels and the small (<= 20 x 20) matrix
// exponential on device.
//
// Replaces (reference file:line):
//   krylov_expm_exec      pytdscf/_integrator.py:453-655 (short_iterative_lanczos), :287-432 (short_iterative_arnoldi)
//   k_krylov_small_expm   pytdscf/_integrator.py:617-637, :401-409 (eigh_tridiagonal / eig + solve on the host CPU)
//   k_lanczos_*           pytdscf/_integrator.py:556-568 ; k_arnoldi_* :247-260 ; k_combine :636-637, :647
//
// Reference quirks reproduced on purpose (SURVEY F2/F3, Appendix B): alpha_l = <v0 | Op v_l> (always the first
// Krylov vector as bra); real parts of alpha are used while every |Im alpha| <= 1e-10; the matvec of iteration 0
// acts on the un-normalised input; stop rule |y_k - y_{k-1}| < thresh evaluated only after the warm-up
// iterations; result re-normalised (conserve_norm) or multiplied back by |psi| (otherwise).
//
// The host loop needs three scalars per iteration (beta_l, |y_k - y_{k-1}|, "alpha is real" flag); they are
// read through a pinned mailbox with one stream synchronisation.  All vector arithmetic stays on device and
// every reduction is a fixed-order two-level tree (deterministic run to run).
#include <cooperative_groups.h>
#include <type_traits>

#include "contract.cuh"

namespace tdvp {

namespace {

constexpr int KCAP = 20;          // Krylov cap, _integrator.py:182
constexpr double EPS_K = 1e-12;   // _integrator.py:22
constexpr int RED_THREADS = 256;
constexpr int RED_MAX_BLOCKS = 592;  // 4 per SM
constexpr int HLD = KCAP + 1;        // leading dimension of the Hessenberg matrix

// mailbox layout inside Handle::d_scal (doubles)
enum : int {
  S_ALPHA = 0,            // alpha[l] complex: 2*l, 2*l+1          (42)
  S_BETA = 64,            // beta[l]                               (21)
  S_ERR = 96,             // |y - prev|^2 -> sqrt
  S_YNORM = 97,           // |y|
  S_B0 = 98,              // |psi| of the input
  S_AREAL = 99,           // 1.0 while every |Im alpha| <= 1e-10
  S_COEF = 128,           // Ritz coefficients c[k] complex          (42)
  S_HESS = 256,           // Arnoldi Hessenberg, complex, HLD x KCAP (882)
  S_TMP = 1280,
};

inline int red_blocks(long long n) {
  long long b = (n + RED_THREADS * 4 - 1) / (RED_THREADS * 4);
  if (b < 1) b = 1;
  if (b > RED_MAX_BLOCKS) b = RED_MAX_BLOCKS;
  return (int)b;
}

// Block-level sum of NV per-thread values, then a fixed-order second level executed by the last block
// to finish ("ticket" pattern).  Returns true in the finishing block with the totals in out_smem[0..NV).
template <int NV>
__device__ bool reduce_all(double (&v)[NV], double* __restrict__ partial, unsigned int* counter, double* out_smem) {
  __shared__ double sm[32][NV + 1];
  __shared__ bool is_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    double x = v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0) sm[warp][i] = x;
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      double x = lane < nwarp ? sm[lane][i] : 0.0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
      if (lane == 0) partial[(size_t)blockIdx.x * NV + i] = x;
    }
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int t = atomicAdd(counter, 1u);
    is_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return false;
  __threadfence();
  // fixed-order reduction of the per-block partials
  double acc[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) acc[i] = 0.0;
  for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) {
#pragma unroll
    for (int i = 0; i < NV; ++i) acc[i] += partial[(size_t)b * NV + i];
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    double x = acc[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0) sm[warp][i] = x;
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      double x = lane < nwarp ? sm[lane][i] : 0.0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
      if (lane == 0) out_smem[i] = x;
    }
  }
  if (threadIdx.x == 0) *counter = 0u;
  __syncthreads();
  return true;
}

// out2 = sum conj(x) * y (conj != 0) or sum x * y
__global__ void __launch_bounds__(RED_THREADS) k_dot(const c128* __restrict__ x, const c128* __restrict__ y, long long n,
                                                      int conj, double* partial, unsigned int* counter, double* out2) {
  __shared__ double tot[2];
  double v[2] = {0.0, 0.0};
  const double s = conj ? -1.0 : 1.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const c128 a = x[i], b = y[i];
    const double ay = s * a.y;
    v[0] += a.x * b.x - ay * b.y;
    v[1] += a.x * b.y + ay * b.x;
  }
  if (reduce_all<2>(v, partial, counter, tot) && threadIdx.x == 0) { out2[0] = tot[0]; out2[1] = (conj == 2) ? 0.0 : tot[1]; }
}

// |x| -> out[0]
__global__ void __launch_bounds__(RED_THREADS) k_norm(const c128* __restrict__ x, long long n, double* partial,
                                                       unsigned int* counter, double* out) {
  __shared__ double tot[1];
  double v[1] = {0.0};
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const c128 a = x[i];
    v[0] += a.x * a.x + a.y * a.y;
  }
  if (reduce_all<1>(v, partial, counter, tot) && threadIdx.x == 0) out[0] = sqrt(tot[0]);
}

// y = x * (mul ? *scal : 1 / *scal)    (scal read from device memory; y may alias x)
__global__ void k_scale_dev(const c128* __restrict__ x, c128* __restrict__ y, long long n, const double* scal, int mul,
                            double min_div) {
  const double s = *scal;
  if (!mul && s < min_div) return;  // Krylov space exhausted: vector is left untouched (it is never used)
  const double f = mul ? s : 1.0 / s;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    c128 a = x[i];
    if (mul) { a.x *= f; a.y *= f; } else { a.x /= s; a.y /= s; }
    y[i] = a;
  }
}

// Lanczos three-term update:  alpha = <v0|w>;  (separate kernel k_dot)   w -= alpha*v1 + beta_prev*v2 ;  beta = |w|
__global__ void __launch_bounds__(RED_THREADS) k_lanczos_update(c128* __restrict__ w, const c128* __restrict__ v1,
                                                                 const c128* __restrict__ v2, long long n,
                                                                 const double* alpha2, const double* beta_prev,
                                                                 double* partial, unsigned int* counter, double* beta_out,
                                                                 double* areal_flag) {
  __shared__ double tot[1];
  const double ar = alpha2[0], ai = alpha2[1];
  const double bp = v2 ? *beta_prev : 0.0;
  double v[1] = {0.0};
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    c128 x = w[i];
    const c128 a = v1[i];
    x.x -= a.x * ar - a.y * ai;
    x.y -= a.x * ai + a.y * ar;
    if (v2) {
      const c128 b = v2[i];
      x.x -= b.x * bp;
      x.y -= b.y * bp;
    }
    w[i] = x;
    v[0] += x.x * x.x + x.y * x.y;
  }
  if (reduce_all<1>(v, partial, counter, tot) && threadIdx.x == 0) {
    beta_out[0] = sqrt(tot[0]);
    if (fabs(ai) > 1e-10) *areal_flag = 0.0;
  }
}

// Small vectors (N <= FUSED_MAX_N: the D <= 64 regime, where a sweep is bound by kernel launches, not bandwidth): the
// three Lanczos vector kernels of one iteration -- alpha = <v0|w>; w -= alpha v_l + beta_{l-1} v_{l-1}, beta = |w|;
// w /= beta -- as ONE kernel run by a single 8-CTA cluster.  Every thread keeps its (at most 8) elements of w in
// registers across the three phases; the two reductions go through distributed shared memory (each CTA publishes its
// partial, cluster barrier, everybody sums the 8 partials in rank order: deterministic).  One SM alone cannot do this:
// it pulls ~150 GB/s from L2 and took 27 us for the 4 MB of traffic (first version of this kernel, r2 c2 profile).
constexpr int FUSED_CLUSTER = 8;    // portable cluster size
constexpr int FUSED_THREADS = 512;
constexpr int FUSED_PER_THREAD = 8;
constexpr long long FUSED_MAX_N = (long long)FUSED_CLUSTER * FUSED_THREADS * FUSED_PER_THREAD;   // 32768

__device__ __forceinline__ void cta_sum2(double& a, double& b, double (*sm)[2]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
  __syncthreads();
  if (lane == 0) { sm[warp][0] = a; sm[warp][1] = b; }
  __syncthreads();
  double ta = 0.0, tb = 0.0;
  for (int w = 0; w < nw; ++w) { ta += sm[w][0]; tb += sm[w][1]; }
  a = ta; b = tb;
}

__global__ void __cluster_dims__(FUSED_CLUSTER, 1, 1) __launch_bounds__(FUSED_THREADS)
    k_lanczos_step_small(const c128* __restrict__ v0, c128* __restrict__ w, const c128* __restrict__ v1,
                         const c128* __restrict__ v2, int n, double* alpha2, const double* beta_prev, double* beta_out,
                         double* areal_flag, double min_div) {
  namespace cgx = cooperative_groups;
  cgx::cluster_group cluster = cgx::this_cluster();
  __shared__ double sm[FUSED_THREADS / 32][2];
  __shared__ double part[2][2];                      // this CTA's partial sums: [phase][re | im]
  const int rank = (int)cluster.block_rank();
  const int base = rank * FUSED_THREADS + threadIdx.x;
  constexpr int STRIDE = FUSED_CLUSTER * FUSED_THREADS;
  c128 x[FUSED_PER_THREAD];
  double ar = 0.0, ai = 0.0;
#pragma unroll
  for (int k = 0; k < FUSED_PER_THREAD; ++k) {
    const int i = base + k * STRIDE;
    x[k] = {0.0, 0.0};
    if (i < n) {
      x[k] = w[i];
      const c128 a = v0[i];
      ar += a.x * x[k].x + a.y * x[k].y;       // conj(v0) * w
      ai += a.x * x[k].y - a.y * x[k].x;
    }
  }
  cta_sum2(ar, ai, sm);
  if (threadIdx.x == 0) { part[0][0] = ar; part[0][1] = ai; }
  cluster.sync();
  ar = 0.0; ai = 0.0;
#pragma unroll
  for (int q = 0; q < FUSED_CLUSTER; ++q) {
    const double* rp = cluster.map_shared_rank(&part[0][0], q);
    ar += rp[0]; ai += rp[1];
  }
  const double bp = v2 ? *beta_prev : 0.0;
  double nn = 0.0, dummy = 0.0;
#pragma unroll
  for (int k = 0; k < FUSED_PER_THREAD; ++k) {
    const int i = base + k * STRIDE;
    if (i < n) {
      const c128 a = v1[i];
      x[k].x -= a.x * ar - a.y * ai;
      x[k].y -= a.x * ai + a.y * ar;
      if (v2) {
        const c128 b = v2[i];
        x[k].x -= b.x * bp;
        x[k].y -= b.y * bp;
      }
      nn += x[k].x * x[k].x + x[k].y * x[k].y;
    }
  }
  cta_sum2(nn, dummy, sm);
  if (threadIdx.x == 0) part[1][0] = nn;
  cluster.sync();
  nn = 0.0;
#pragma unroll
  for (int q = 0; q < FUSED_CLUSTER; ++q) nn += *cluster.map_shared_rank(&part[1][0], q);
  const double beta = sqrt(nn);
  if (rank == 0 && threadIdx.x == 0) {
    alpha2[0] = ar; alpha2[1] = ai;
    beta_out[0] = beta;
    if (fabs(ai) > 1e-10) *areal_flag = 0.0;
  }
  const bool scale = beta >= min_div;          // Krylov space exhausted otherwise: the vector is stored unscaled (never used)
#pragma unroll
  for (int k = 0; k < FUSED_PER_THREAD; ++k) {
    const int i = base + k * STRIDE;
    if (i < n) {
      c128 y = x[k];
      if (scale) { y.x /= beta; y.y /= beta; }
      w[i] = y;
    }
  }
  cluster.sync();                              // nobody leaves while a neighbour may still read its partials
}

// Arnoldi: h[i] = <V_i | w>, i < k   (one pass over w, k passes over V)
__global__ void __launch_bounds__(RED_THREADS) k_arnoldi_dots(const c128* __restrict__ V, long long ldv, int k,
                                                               const c128* __restrict__ w, long long n, double* partial,
                                                               unsigned int* counter, double* hcol /* complex, stride 1 */) {
  __shared__ double tot[2 * KCAP];
  double v[2 * KCAP];
#pragma unroll
  for (int i = 0; i < 2 * KCAP; ++i) v[i] = 0.0;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    const c128 b = w[e];
#pragma unroll
    for (int i = 0; i < KCAP; ++i) {
      if (i < k) {
        const c128 a = V[(long long)i * ldv + e];
        v[2 * i] += a.x * b.x + a.y * b.y;
        v[2 * i + 1] += a.x * b.y - a.y * b.x;
      }
    }
  }
  if (reduce_all<2 * KCAP>(v, partial, counter, tot)) {
    for (int i = threadIdx.x; i < 2 * k; i += blockDim.x) hcol[i] = tot[i];
  }
}

// Arnoldi: w -= sum_i h[i] V_i ; beta = |w|
__global__ void __launch_bounds__(RED_THREADS) k_arnoldi_update(const c128* __restrict__ V, long long ldv, int k,
                                                                 c128* __restrict__ w, long long n, const double* hcol,
                                                                 double* partial, unsigned int* counter, double* beta_out) {
  __shared__ double tot[1];
  __shared__ double hs[2 * KCAP];
  for (int i = threadIdx.x; i < 2 * k; i += blockDim.x) hs[i] = hcol[i];
  __syncthreads();
  double v[1] = {0.0};
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    c128 x = w[e];
    double sx = 0.0, sy = 0.0;
    for (int i = 0; i < k; ++i) {
      const c128 a = V[(long long)i * ldv + e];
      sx += hs[2 * i] * a.x - hs[2 * i + 1] * a.y;
      sy += hs[2 * i] * a.y + hs[2 * i + 1] * a.x;
    }
    x.x -= sx;
    x.y -= sy;
    w[e] = x;
    v[0] += x.x * x.x + x.y * x.y;
  }
  if (reduce_all<1>(v, partial, counter, tot) && threadIdx.x == 0) beta_out[0] = sqrt(tot[0]);
}

// y = sum_{i<k} c[i] V_i ;  err = |y - prev| ; ynorm = |y| ; optionally prev <- y is done by pointer swap on host
__global__ void __launch_bounds__(RED_THREADS) k_combine(const c128* __restrict__ V, long long ldv, int k,
                                                          const double* coef, c128* __restrict__ y,
                                                          const c128* __restrict__ prev, long long n, double* partial,
                                                          unsigned int* counter, double* err_out, double* ynorm_out) {
  __shared__ double tot[2];
  __shared__ double cs[2 * KCAP];
  for (int i = threadIdx.x; i < 2 * k; i += blockDim.x) cs[i] = coef[i];
  __syncthreads();
  double v[2] = {0.0, 0.0};
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    double sx = 0.0, sy = 0.0;
    for (int i = 0; i < k; ++i) {
      const c128 a = V[(long long)i * ldv + e];
      sx += cs[2 * i] * a.x - cs[2 * i + 1] * a.y;
      sy += cs[2 * i] * a.y + cs[2 * i + 1] * a.x;
    }
    y[e] = {sx, sy};
    v[1] += sx * sx + sy * sy;
    if (prev) {
      const c128 p = prev[e];
      const double dx = sx - p.x, dy = sy - p.y;
      v[0] += dx * dx + dy * dy;
    }
  }
  if (reduce_all<2>(v, partial, counter, tot) && threadIdx.x == 0) {
    err_out[0] = sqrt(tot[0]);
    ynorm_out[0] = sqrt(tot[1]);
  }
}

// c = expm(scale * T)[:, 0] for the k x k Krylov matrix, one CTA.
//   mode 0: symmetric tridiagonal from alpha (complex, real parts only while *areal != 0) and beta (sub/super diag)
//   mode 1: dense upper Hessenberg `hess` (complex, leading dimension HLD, column l at hess[:, l])
// Scaling-and-squaring Taylor (degree 20 at |A|_1 <= 0.5): truncation ~1e-26, rounding ~ 2^s * eps.
__global__ void __launch_bounds__(512) k_krylov_small_expm(int mode, int k, const double* alpha, const double* beta,
                                                            const double* areal, const double* hess, double scale_re,
                                                            double scale_im, double* coef) {
  __shared__ c128 A[KCAP * KCAP], E[KCAP * KCAP], T[KCAP * KCAP], U[KCAP * KCAP];
  __shared__ double colsum[KCAP];
  __shared__ int s_sq;
  const int tid = threadIdx.x;
  const int kk = k * k;
  const c128 sc = {scale_re, scale_im};
  // "alpha is real" is a property of the k alphas this Ritz step uses (the reference tests them when it builds the matrix,
  // _integrator.py:617-623), not of whatever later iterations a run-ahead stream may already have produced
  __shared__ int s_areal;
  if (tid == 0) {
    int r = 1;
    if (mode == 0)
      for (int i = 0; i < k; ++i)
        if (fabs(alpha[2 * i + 1]) > 1e-10) r = 0;
    s_areal = r;
  }
  __syncthreads();
  (void)areal;
  for (int e = tid; e < kk; e += blockDim.x) {
    const int i = e / k, j = e % k;
    c128 t = {0.0, 0.0};
    if (mode == 0) {
      if (i == j) {
        t.x = alpha[2 * i];
        t.y = s_areal ? 0.0 : alpha[2 * i + 1];
      } else if (i == j + 1) {
        t.x = beta[j];
      } else if (j == i + 1) {
        t.x = beta[i];
      }
    } else {
      t.x = hess[2 * (j * HLD + i)];
      t.y = hess[2 * (j * HLD + i) + 1];
    }
    A[e] = cmul(sc, t);
  }
  __syncthreads();
  if (tid < k) {
    double s = 0.0;
    for (int i = 0; i < k; ++i) s += hypot(A[i * k + tid].x, A[i * k + tid].y);
    colsum[tid] = s;
  }
  __syncthreads();
  if (tid == 0) {
    double nrm = 0.0;
    for (int j = 0; j < k; ++j) nrm = fmax(nrm, colsum[j]);
    int s = 0;
    while (nrm > 0.5 && s < 60) { nrm *= 0.5; ++s; }
    s_sq = s;
  }
  __syncthreads();
  const int s = s_sq;
  const double f = ldexp(1.0, -s);
  for (int e = tid; e < kk; e += blockDim.x) {
    A[e].x *= f; A[e].y *= f;
    const int i = e / k, j = e % k;
    E[e] = {i == j ? 1.0 : 0.0, 0.0};
    T[e] = E[e];
  }
  __syncthreads();
  for (int m = 1; m <= 20; ++m) {  // T <- T*A/m ; E += T
    const double inv = 1.0 / m;
    for (int e = tid; e < kk; e += blockDim.x) {
      const int i = e / k, j = e % k;
      double sx = 0.0, sy = 0.0;
      for (int p = 0; p < k; ++p) {
        const c128 a = T[i * k + p], b = A[p * k + j];
        sx += a.x * b.x - a.y * b.y;
        sy += a.x * b.y + a.y * b.x;
      }
      U[e] = {sx * inv, sy * inv};
    }
    __syncthreads();
    for (int e = tid; e < kk; e += blockDim.x) {
      T[e] = U[e];
      E[e].x += U[e].x;
      E[e].y += U[e].y;
    }
    __syncthreads();
  }
  for (int q = 0; q < s; ++q) {  // E <- E*E
    for (int e = tid; e < kk; e += blockDim.x) {
      const int i = e / k, j = e % k;
      double sx = 0.0, sy = 0.0;
      for (int p = 0; p < k; ++p) {
        const c128 a = E[i * k + p], b = E[p * k + j];
        sx += a.x * b.x - a.y * b.y;
        sy += a.x * b.y + a.y * b.x;
      }
      U[e] = {sx, sy};
    }
    __syncthreads();
    for (int e = tid; e < kk; e += blockDim.x) E[e] = U[e];
    __syncthreads();
  }
  if (tid < k) {
    coef[2 * tid] = E[tid * k].x;
    coef[2 * tid + 1] = E[tid * k].y;
  }
}

// y = sum_{i<k} c[i] V_i for arbitrary k (coefficients read from global memory); err = |y - prev|, ynorm = |y|
__global__ void __launch_bounds__(RED_THREADS) k_combine_big(const c128* __restrict__ V, long long ldv, int k,
                                                              const double* __restrict__ coef, c128* __restrict__ y,
                                                              const c128* __restrict__ prev, long long n, double* partial,
                                                              unsigned int* counter, double* err_out, double* ynorm_out) {
  __shared__ double tot[2];
  double v[2] = {0.0, 0.0};
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    double sx = 0.0, sy = 0.0;
    for (int i = 0; i < k; ++i) {
      const c128 a = V[(long long)i * ldv + e];
      const double cr = __ldg(&coef[2 * i]), ci = __ldg(&coef[2 * i + 1]);
      sx += cr * a.x - ci * a.y;
      sy += cr * a.y + ci * a.x;
    }
    y[e] = {sx, sy};
    v[1] += sx * sx + sy * sy;
    if (prev) {
      const c128 p = prev[e];
      const double dx = sx - p.x, dy = sy - p.y;
      v[0] += dx * dx + dy * dy;
    }
  }
  if (reduce_all<2>(v, partial, counter, tot) && threadIdx.x == 0) {
    err_out[0] = sqrt(tot[0]);
    ynorm_out[0] = sqrt(tot[1]);
  }
}

// Eigenvector of the real symmetric tridiagonal matrix (diag a[0..k), off-diagonal b[0..k-1)) for its smallest
// (root == 0) or largest (root != 0) eigenvalue: Sturm-sequence bisection + inverse iteration, one thread
// (k is the Lanczos dimension).  Sign convention: positive component along the first Lanczos vector.
// (The reference calls scipy.linalg.eigh_tridiagonal, whose eigenvector sign is LAPACK-internal and unpinned.)
__global__ void k_tridiag_eigvec(int k, const double* __restrict__ a, const double* __restrict__ b, int root,
                                 double* __restrict__ coef, double* __restrict__ work) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (k == 1) { coef[0] = 1.0; coef[1] = 0.0; return; }
  double lo = a[0], hi = a[0], nrm = 0.0;
  for (int i = 0; i < k; ++i) {
    const double r = (i > 0 ? fabs(b[i - 1]) : 0.0) + (i < k - 1 ? fabs(b[i]) : 0.0);
    lo = fmin(lo, a[i] - r);
    hi = fmax(hi, a[i] + r);
    nrm = fmax(nrm, fabs(a[i]) + r);
  }
  const int target = root == 0 ? 1 : k;  // find lambda with count(lambda) >= target, i.e. the target-th smallest
  const double tiny = 2.3e-308 / 2.2e-16;
  for (int it = 0; it < 200; ++it) {
    const double mid = 0.5 * (lo + hi);
    if (mid <= lo || mid >= hi) break;
    int cnt = 0;
    double q = a[0] - mid;
    if (q < 0.0) ++cnt;
    for (int i = 1; i < k; ++i) {
      if (fabs(q) < tiny) q = (q < 0.0 ? -tiny : tiny);
      q = a[i] - mid - b[i - 1] * b[i - 1] / q;
      if (q < 0.0) ++cnt;
    }
    if (cnt >= target) hi = mid; else lo = mid;
  }
  const double lam = 0.5 * (lo + hi);
  // inverse iteration on (T - lam I) with partial pivoting (tridiagonal LU, fill-in in du2)
  double* dl = work;            // sub-diagonal multipliers   (k-1)
  double* dd = work + k;        // diagonal                   (k)
  double* du = work + 2 * k;    // first super-diagonal       (k-1)
  double* du2 = work + 3 * k;   // second super-diagonal      (k-2)
  double* x = work + 4 * k;     // solution                   (k)
  int* piv = reinterpret_cast<int*>(work + 5 * k);
  const double shift = lam + (root == 0 ? -1.0 : 1.0) * 4.0 * 2.2e-16 * fmax(nrm, 1e-300);
  for (int i = 0; i < k; ++i) { dd[i] = a[i] - shift; x[i] = 1.0 / sqrt((double)k); }
  for (int i = 0; i < k - 1; ++i) { dl[i] = b[i]; du[i] = b[i]; }
  for (int i = 0; i < k - 2; ++i) du2[i] = 0.0;
  for (int i = 0; i < k - 1; ++i) {
    if (fabs(dd[i]) >= fabs(dl[i])) {
      piv[i] = 0;
      if (dd[i] == 0.0) dd[i] = 2.2e-16 * fmax(nrm, 1e-300);
      const double f = dl[i] / dd[i];
      dl[i] = f;
      dd[i + 1] -= f * du[i];
      if (i < k - 2) du2[i] = 0.0;
    } else {
      piv[i] = 1;
      const double f = dd[i] / dl[i];
      dd[i] = dl[i];
      dl[i] = f;
      const double t = du[i];
      du[i] = dd[i + 1];
      dd[i + 1] = t - f * du[i];
      if (i < k - 2) { du2[i] = du[i + 1]; du[i + 1] = -f * du[i + 1]; }
    }
  }
  if (dd[k - 1] == 0.0) dd[k - 1] = 2.2e-16 * fmax(nrm, 1e-300);
  for (int iter = 0; iter < 4; ++iter) {
    for (int i = 0; i < k - 1; ++i) {        // forward: apply L^-1 with the row interchanges
      if (piv[i]) { const double t = x[i]; x[i] = x[i + 1]; x[i + 1] = t - dl[i] * x[i]; }
      else x[i + 1] -= dl[i] * x[i];
    }
    x[k - 1] /= dd[k - 1];                   // backward: U x = y
    if (k > 1) x[k - 2] = (x[k - 2] - du[k - 2] * x[k - 1]) / dd[k - 2];
    for (int i = k - 3; i >= 0; --i) x[i] = (x[i] - du[i] * x[i + 1] - du2[i] * x[i + 2]) / dd[i];
    double s = 0.0;
    for (int i = 0; i < k; ++i) s += x[i] * x[i];
    s = 1.0 / sqrt(s);
    for (int i = 0; i < k; ++i) x[i] *= s;
  }
  const double sg = x[0] < 0.0 ? -1.0 : 1.0;
  for (int i = 0; i < k; ++i) { coef[2 * i] = sg * x[i]; coef[2 * i + 1] = 0.0; }
}

__global__ void k_set_scalars(double* p, int n, double v) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) p[i] = v;
}

__global__ void k_store_beta_hess(double* hess, int l, const double* beta) {
  // hess[l+1, l] = beta (real)
  hess[2 * (l * HLD + (l + 1))] = *beta;
  hess[2 * (l * HLD + (l + 1)) + 1] = 0.0;
}

int lc(Handle* h, const char* what) {
  count_launch();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(h, e, what, __FILE__, __LINE__);
  return 0;
}

}  // namespace

int inner_exec(Handle* h, long long n, const c128* bra, const c128* ket, int conj, c128* host_out) {
  { ProfScope _ps(h->stream, "vec.k_dot"); k_dot<<<red_blocks(n), RED_THREADS, 0, h->stream>>>(bra, ket, n, conj, h->d_partial, h->d_counter, h->d_scal + S_TMP); }
  TDVP_TRY(lc(h, "k_dot"));
  TDVP_CUDA(h, cudaMemcpyAsync(h->h_scal + S_TMP, h->d_scal + S_TMP, 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  TDVP_CUDA(h, cudaStreamSynchronize(h->stream));
  host_out->x = h->h_scal[S_TMP];
  host_out->y = h->h_scal[S_TMP + 1];
  return 0;
}

namespace {

// exp(scale * Op) psi for an operator given as `apply(x, y)`: y = Op x on vectors of N elements; `contr` = workspace
// elements the operator needs per application.  `checked`: report a workspace the device cannot hold as
// TDVP_ERR_NO_MEMORY (the two-site solve, whose basis can outgrow the device).
template <class Apply>
int krylov_expm_core(Handle* h, int kind, double scale_re, double scale_im, double thresh, int n_warmup, int conserve_norm,
                     long long N, size_t contr, bool checked, Apply&& apply, c128* psi, int* niter) {
  // The reference sizes the Krylov space (cap, warm-up bound, "space exhausted" test) by the tensor it was GIVEN; with
  // adaptive bond growth that tensor is smaller than the zero-extended vector the recurrence runs on
  // (_integrator.py:178-186, 524, 570): tdvp_set_krylov_size passes that size for the next solve.
  const long long Nref = (h->krylov_size_override > 0 && h->krylov_size_override < N) ? h->krylov_size_override : N;
  h->krylov_size_override = 0;
  const int ndim = (int)(Nref < KCAP ? Nref : KCAP);
  int n_warm = n_warmup;
  if (n_warm > Nref) n_warm = (int)Nref;
  if (n_warm < 0) n_warm = 0;

  // ---- workspace: V[(ndim+1) x N], y, prev, + contraction scratch ----
  const size_t need = sizeof(c128) * ((size_t)(ndim + 3) * N + contr) + 256 * 16;
  if (checked) TDVP_TRY(ws_reserve_checked(h, need, "krylov_expm2 (Krylov basis)"));
  else TDVP_TRY(ws_reserve(h, need));
  c128* V = (c128*)ws_alloc(h, sizeof(c128) * (size_t)(ndim + 1) * N);
  c128* ybuf[2] = {(c128*)ws_alloc(h, sizeof(c128) * N), (c128*)ws_alloc(h, sizeof(c128) * N)};
  if (!V || !ybuf[0] || !ybuf[1]) { set_error(h, "krylov_expm: workspace"); return TDVP_ERR_ARG; }
  double* S = h->d_scal;
  cudaStream_t st = h->stream;
  const int nb = red_blocks(N);
  const int vb = nb;

  auto matvec = [&](const c128* x, c128* y) -> int {
    ++h->krylov_matvecs;
    return apply(x, y);
  };

  // ---- v0 ----
  { ProfScope _ps(st, "vec.k_set_scalars"); k_set_scalars<<<1, 32, 0, st>>>(S + S_AREAL, 1, 1.0); }
  TDVP_TRY(lc(h, "k_set_scalars"));
  TDVP_CUDA(h, cudaMemcpyAsync(V, psi, sizeof(c128) * N, cudaMemcpyDeviceToDevice, st));
  if (!conserve_norm) {
    { ProfScope _ps(st, "vec.k_norm"); k_norm<<<nb, RED_THREADS, 0, st>>>(V, N, h->d_partial, h->d_counter, S + S_B0); }
    TDVP_TRY(lc(h, "k_norm"));
    TDVP_CUDA(h, cudaMemcpyAsync(h->h_scal + S_B0, S + S_B0, sizeof(double), cudaMemcpyDeviceToHost, st));
    TDVP_CUDA(h, cudaStreamSynchronize(st));
    if (h->h_scal[S_B0] == 0.0) { set_error(h, "Initial psi has zero norm."); return TDVP_ERR_ZERO_NORM; }
    { ProfScope _ps(st, "vec.k_scale_dev"); k_scale_dev<<<vb, RED_THREADS, 0, st>>>(V, V, N, S + S_B0, 0, 0.0); }
    TDVP_TRY(lc(h, "k_scale_dev"));
  }
  ++h->krylov_solves;

  int cur = 0;          // ybuf[cur] receives the next Ritz vector
  bool have_prev = false;
  int nvec = 1;         // Krylov vectors stored (Arnoldi may stop appending)
  int synced = 0;       // beta_[0 .. synced) are known on the host
  bool side_pending = false;   // a Ritz step is in flight on the side stream (ev_side marks its end)
  for (int l = 0; l < ndim; ++l) {
    c128* w = V + (size_t)(kind == TDVP_KRYLOV_ARNOLDI ? nvec : l + 1) * N;
    const c128* src = (l == 0) ? psi : (kind == TDVP_KRYLOV_ARNOLDI ? V + (size_t)(nvec - 1) * N : V + (size_t)l * N);
    TDVP_TRY(matvec(src, w));
    if (!conserve_norm && l == 0) {
      { ProfScope _ps(st, "vec.k_scale_dev"); k_scale_dev<<<vb, RED_THREADS, 0, st>>>(w, w, N, S + S_B0, 0, 0.0); }
      TDVP_TRY(lc(h, "k_scale_dev"));
    }
    if (kind == TDVP_KRYLOV_LANCZOS_REF && N <= FUSED_MAX_N) {
      { ProfScope _ps(st, "vec.k_lanczos_step_small");
        k_lanczos_step_small<<<FUSED_CLUSTER, FUSED_THREADS, 0, st>>>(V, w, V + (size_t)l * N, l > 0 ? V + (size_t)(l - 1) * N : nullptr, (int)N,
                                                           S + S_ALPHA + 2 * l, S + S_BETA + (l > 0 ? l - 1 : 0), S + S_BETA + l,
                                                           S + S_AREAL, EPS_K); }
      TDVP_TRY(lc(h, "k_lanczos_step_small"));
    } else if (kind == TDVP_KRYLOV_LANCZOS_REF) {
      { ProfScope _ps(st, "vec.k_dot"); k_dot<<<nb, RED_THREADS, 0, st>>>(V, w, N, 1, h->d_partial, h->d_counter, S + S_ALPHA + 2 * l); }
      TDVP_TRY(lc(h, "k_dot"));
      { ProfScope _ps(st, "vec.k_lanczos_update"); k_lanczos_update<<<nb, RED_THREADS, 0, st>>>(w, V + (size_t)l * N, l > 0 ? V + (size_t)(l - 1) * N : nullptr, N,
                                                     S + S_ALPHA + 2 * l, S + S_BETA + (l > 0 ? l - 1 : 0), h->d_partial,
                                                     h->d_counter, S + S_BETA + l, S + S_AREAL); }
      TDVP_TRY(lc(h, "k_lanczos_update"));
    } else {
      double* hcol = S + S_HESS + 2 * (l * HLD);
      { ProfScope _ps(st, "vec.k_arnoldi_dots"); k_arnoldi_dots<<<nb, RED_THREADS, 0, st>>>(V, N, nvec, w, N, h->d_partial, h->d_counter, hcol); }
      TDVP_TRY(lc(h, "k_arnoldi_dots"));
      { ProfScope _ps(st, "vec.k_arnoldi_update"); k_arnoldi_update<<<nb, RED_THREADS, 0, st>>>(V, N, nvec, w, N, hcol, h->d_partial, h->d_counter, S + S_BETA + l); }
      TDVP_TRY(lc(h, "k_arnoldi_update"));
      if (l + 1 < HLD) {
        { ProfScope _ps(st, "vec.k_store_beta_hess"); k_store_beta_hess<<<1, 1, 0, st>>>(S + S_HESS, l, S + S_BETA + l); }
        TDVP_TRY(lc(h, "k_store_beta_hess"));
      }
    }
    // w /= beta when beta >= EPS (Lanczos) / > EPS (Arnoldi): decided on device, mirrored on host at the next read-back
    if (!(kind == TDVP_KRYLOV_LANCZOS_REF && N <= FUSED_MAX_N)) {   // (the fused small-N kernel has done it already)
      { ProfScope _ps(st, "vec.k_scale_dev"); k_scale_dev<<<vb, RED_THREADS, 0, st>>>(w, w, N, S + S_BETA + l, 0, kind == TDVP_KRYLOV_ARNOLDI ? nextafter(EPS_K, 1.0) : EPS_K); }
      TDVP_TRY(lc(h, "k_scale_dev"));
    }
    // Warm-up iterations (the reference skips the Ritz step there, _integrator.py:560-575) need nothing on the host:
    // the beta values are read back together with the first convergence scalar, so the stream keeps running ahead.
    // A breakdown (beta < eps) inside the warm-up is detected at that read-back and replayed from the stored basis.
    if (l < n_warm && (long long)(l + 1) < Nref) {
      if (kind == TDVP_KRYLOV_ARNOLDI) ++nvec;    // speculative: beta > eps (checked below)
      continue;
    }

    // ---- Ritz step on device ----
    const int k = l + 1;
    auto ritz_on = [&](cudaStream_t rs, double* partial, unsigned int* counter, int kk, c128* yout, const c128* yprev) -> int {
      if (kind == TDVP_KRYLOV_LANCZOS_REF)
        { ProfScope _ps(rs, "vec.k_krylov_small_expm"); k_krylov_small_expm<<<1, 512, 0, rs>>>(0, kk, S + S_ALPHA, S + S_BETA, S + S_AREAL, nullptr, scale_re, scale_im, S + S_COEF); }
      else
        { ProfScope _ps(rs, "vec.k_krylov_small_expm"); k_krylov_small_expm<<<1, 512, 0, rs>>>(1, kk, nullptr, nullptr, nullptr, S + S_HESS, scale_re, scale_im, S + S_COEF); }
      TDVP_TRY(lc(h, "k_krylov_small_expm"));
      { ProfScope _ps(rs, "vec.k_combine"); k_combine<<<nb, RED_THREADS, 0, rs>>>(V, N, kk, S + S_COEF, yout, yprev, N, partial, counter, S + S_ERR, S + S_YNORM); }
      return lc(h, "k_combine");
    };
    // Ritz step on the main stream (after whatever the side stream still has in flight: it shares S_COEF / S_ERR)
    auto ritz = [&](int kk, c128* yout, const c128* yprev) -> int {
      if (side_pending) { TDVP_CUDA(h, cudaStreamWaitEvent(st, h->ev_side, 0)); side_pending = false; }
      return ritz_on(st, h->d_partial, h->d_counter, kk, yout, yprev);
    };
    auto finish = [&](c128* yfin, int iters) -> int {
      // rescale: y / |y| (conserve_norm) or y * b0, written back into psi
      if (conserve_norm) { ProfScope _ps(st, "vec.k_scale_dev"); k_scale_dev<<<vb, RED_THREADS, 0, st>>>(yfin, psi, N, S + S_YNORM, 0, 0.0); }
      else { ProfScope _ps(st, "vec.k_scale_dev"); k_scale_dev<<<vb, RED_THREADS, 0, st>>>(yfin, psi, N, S + S_B0, 1, 0.0); }
      TDVP_TRY(lc(h, "k_scale_dev"));
      if (niter) *niter = iters;
      return 0;
    };
    c128* y = ybuf[cur];
    const c128* prev = have_prev ? ybuf[cur ^ 1] : nullptr;
    // The first checked iteration cannot stop on the change of the Ritz vector (there is no previous one): only on a
    // breakdown (beta < eps), which the next read-back detects and replays from the stored basis exactly like a breakdown
    // inside the warm-up.  So nothing is read back here; the Ritz vector (needed as "previous" by the next check) is
    // formed on the side stream while the main stream goes on with the next matvec.
    if (!have_prev && (long long)(l + 1) < Nref && l + 1 < ndim && h->side) {
      TDVP_CUDA(h, cudaEventRecord(h->ev_main, st));
      TDVP_CUDA(h, cudaStreamWaitEvent(h->side, h->ev_main, 0));
      TDVP_TRY(ritz_on(h->side, h->d_partial_side, h->d_counter_side, k, y, nullptr));
      TDVP_CUDA(h, cudaEventRecord(h->ev_side, h->side));
      side_pending = true;
      if (kind == TDVP_KRYLOV_ARNOLDI) ++nvec;    // speculative, as in the warm-up
      have_prev = true;
      cur ^= 1;
      continue;
    }
    TDVP_TRY(ritz(k, y, prev));
    // one read-back per checked iteration: beta_[synced .. l] and the change of the Ritz vector
    TDVP_CUDA(h, cudaMemcpyAsync(h->h_scal + S_BETA + synced, S + S_BETA + synced, sizeof(double) * (l + 1 - synced), cudaMemcpyDeviceToHost, st));
    TDVP_CUDA(h, cudaMemcpyAsync(h->h_scal + S_ERR, S + S_ERR, sizeof(double), cudaMemcpyDeviceToHost, st));
    TDVP_CUDA(h, cudaStreamSynchronize(st));
    for (int j = synced; j <= l; ++j) {
      const double bj = h->h_scal[S_BETA + j];
      if (!(bj == bj)) { set_error(h, "krylov_expm: NaN encountered in the Krylov recurrence"); return TDVP_ERR_NOT_CONVERGED; }
      if (j < l && bj < EPS_K) {
        // the recurrence broke down at warm-up iteration j: the reference stops there with a (j+1)-vector Ritz step
        TDVP_TRY(ritz(j + 1, y, nullptr));
        return finish(y, j + 1);
      }
    }
    synced = l + 1;
    const double beta = h->h_scal[S_BETA + l];
    const bool conv = beta < EPS_K || (long long)(l + 1) == Nref;
    if (kind == TDVP_KRYLOV_ARNOLDI && beta > EPS_K) ++nvec;
    const bool done = conv || (have_prev && h->h_scal[S_ERR] < thresh);
    if (done) return finish(y, l + 1);
    have_prev = true;
    cur ^= 1;
  }
  set_error(h, kind == TDVP_KRYLOV_ARNOLDI ? "Short Iterative Arnoldi is not converged in 20 basis"
                                           : "Short Iterative Lanczos is not converged. Try shorter time interval.");
  return TDVP_ERR_NOT_CONVERGED;
}

}  // namespace

int krylov_expm_exec(Handle* h, int kind, double scale_re, double scale_im, double thresh, int n_warmup,
                     int conserve_norm, const tdvp_heff_term* hterms, const tdvp_keff_term* kterms, int nterms,
                     int Dl, int d, int Dr, c128* psi, int* niter) {
  if ((hterms == nullptr) == (kterms == nullptr)) { set_error(h, "krylov_expm: pass exactly one of hterms / kterms"); return TDVP_ERR_ARG; }
  if (kind != TDVP_KRYLOV_LANCZOS_REF && kind != TDVP_KRYLOV_ARNOLDI) { set_error(h, "krylov_expm: bad kind"); return TDVP_ERR_ARG; }
  const bool isH = hterms != nullptr;
  const long long N = isH ? (long long)Dl * d * Dr : (long long)Dl * Dr;
  if (N <= 0) { set_error(h, "krylov_expm: empty vector"); return TDVP_ERR_SHAPE; }
  const size_t contr = isH ? heff_ws_elems(hterms, nterms, Dl, d, Dr) : keff_ws_elems(kterms, nterms, Dl, Dr);
  return krylov_expm_core(h, kind, scale_re, scale_im, thresh, n_warmup, conserve_norm, N, contr, false,
                          [&](const c128* x, c128* y) {
                            return isH ? heff_apply_exec(h, hterms, nterms, Dl, d, Dr, x, y)
                                       : keff_apply_exec(h, kterms, nterms, Dl, Dr, x, y);
                          },
                          psi, niter);
}

// Two-site operator: theta(Dl, d1, d2, Dr), the same solver on the heff2 chain.
int krylov_expm2_exec(Handle* h, int kind, double scale_re, double scale_im, double thresh, int n_warmup,
                      int conserve_norm, const tdvp_heff2_term* terms, int nterms, int Dl, int d1, int d2, int Dr, c128* theta,
                      int* niter) {
  if (kind != TDVP_KRYLOV_LANCZOS_REF && kind != TDVP_KRYLOV_ARNOLDI) { set_error(h, "krylov_expm2: bad kind"); return TDVP_ERR_ARG; }
  const long long N = (long long)Dl * d1 * d2 * Dr;
  const size_t contr = heff2_ws_elems(terms, nterms, Dl, d1, d2, Dr);
  return krylov_expm_core(h, kind, scale_re, scale_im, thresh, n_warmup, conserve_norm, N, contr, true,
                          [&](const c128* x, c128* y) { return heff2_apply_exec(h, terms, nterms, Dl, d1, d2, Dr, x, y); },
                          theta, niter);
}

// Lowest (root = 0) / highest eigenvector of the effective Hamiltonian by textbook Lanczos -- the site solve of
// improved relaxation (pytdscf/_integrator.py:74-138, matrix_diagonalize_lanczos): alpha_i = Re<v_i|H v_i>, full
// three-term recurrence, Ritz vector rebuilt every iteration, stop on |y_i - y_{i-1}| < thresh, beta < 1e-12 or
// i == N.  The result is normalised (pytdscf/_mps_cls.py:1078-1084).
int lanczos_eigvec_exec(Handle* h, const tdvp_heff_term* hterms, int nterms, int Dl, int d, int Dr, c128* psi, int root,
                        double thresh, int* niter) {
  const long long N = (long long)Dl * d * Dr;
  if (N <= 0) { set_error(h, "lanczos_eigvec: empty vector"); return TDVP_ERR_SHAPE; }
  // Lanczos basis: the reference stores every vector (up to 3000).  The workspace starts with room for 32 and doubles on
  // demand (contents preserved), bounded by 3000, N and half of the free device memory.
  const long long kabs = N < 3000 ? N : 3000;
  size_t free_b = 0, total_b = 0;
  TDVP_CUDA(h, cudaMemGetInfo(&free_b, &total_b));
  long long mem_cap = (long long)((free_b / 2 + h->ws_bytes) / (sizeof(c128) * (size_t)N)) - 8;
  if (mem_cap < 4) mem_cap = 4;
  const long long klimit = kabs < mem_cap ? kabs : mem_cap;
  long long kmax = klimit < 32 ? klimit : 32;
  const size_t contr = heff_ws_elems(hterms, nterms, Dl, d, Dr);
  auto bytes_for = [&](long long k) {
    return sizeof(c128) * ((size_t)(k + 4) * N + contr) + sizeof(double) * (size_t)(10 * kabs + 64) + 256 * 16;
  };
  TDVP_TRY(ws_reserve(h, bytes_for(kmax)));
  // small arrays first (sized for the absolute cap), the growing basis last
  double* alpha = (double*)ws_alloc(h, sizeof(double) * (size_t)(kabs + 2));   // real diagonal
  double* beta = (double*)ws_alloc(h, sizeof(double) * (size_t)(kabs + 2));    // beta[i] = |w_i|, off-diagonal i
  double* coef = (double*)ws_alloc(h, sizeof(double) * 2 * (size_t)(kabs + 2));
  double* work = (double*)ws_alloc(h, sizeof(double) * 6 * (size_t)(kabs + 2));
  c128* ybuf[2] = {(c128*)ws_alloc(h, sizeof(c128) * N), (c128*)ws_alloc(h, sizeof(c128) * N)};
  const size_t top_before_V = h->ws_top;
  c128* V = (c128*)ws_alloc(h, sizeof(c128) * (size_t)(kmax + 2) * N);
  if (!V || !ybuf[0] || !ybuf[1] || !alpha || !beta || !coef || !work) { set_error(h, "lanczos_eigvec: workspace"); return TDVP_ERR_ARG; }
  double* S = h->d_scal;
  cudaStream_t st = h->stream;
  const int nb = red_blocks(N);
  TDVP_CUDA(h, cudaMemcpyAsync(V, psi, sizeof(c128) * N, cudaMemcpyDeviceToDevice, st));
  ++h->krylov_solves;
  int cur = 0;
  bool have_prev = false;
  for (long long i = 0; i <= klimit; ++i) {
    if (i == kmax && kmax < klimit) {
      // basis full: double it, keeping everything already stored (pointers are rebased onto the new buffer)
      long long knew = 2 * kmax < klimit ? 2 * kmax : klimit;
      const unsigned char* old_base = h->ws;
      TDVP_TRY(ws_grow_preserve(h, bytes_for(knew)));
      const ptrdiff_t delta = h->ws - old_base;
      auto rebase = [&](auto*& p) { p = reinterpret_cast<std::remove_reference_t<decltype(p)>>(reinterpret_cast<unsigned char*>(p) + delta); };
      rebase(alpha); rebase(beta); rebase(coef); rebase(work); rebase(ybuf[0]); rebase(ybuf[1]); rebase(V);
      h->ws_top = top_before_V;
      if (!ws_alloc(h, sizeof(c128) * (size_t)(knew + 2) * N)) { set_error(h, "lanczos_eigvec: workspace"); return TDVP_ERR_ARG; }
      kmax = knew;
    }
    c128* vi = V + (size_t)i * N;
    c128* w = V + (size_t)(i + 1) * N;
    ++h->krylov_matvecs;
    TDVP_TRY(heff_apply_exec(h, hterms, nterms, Dl, d, Dr, vi, w));
    { ProfScope _ps(st, "vec.k_dot"); k_dot<<<nb, RED_THREADS, 0, st>>>(vi, w, N, 2, h->d_partial, h->d_counter, S + S_TMP); }
    TDVP_TRY(lc(h, "k_dot"));
    TDVP_CUDA(h, cudaMemcpyAsync(alpha + i, S + S_TMP, sizeof(double), cudaMemcpyDeviceToDevice, st));
    { ProfScope _ps(st, "vec.k_lanczos_update");
      k_lanczos_update<<<nb, RED_THREADS, 0, st>>>(w, vi, i > 0 ? V + (size_t)(i - 1) * N : nullptr, N, S + S_TMP,
                                                     i > 0 ? beta + (i - 1) : beta, h->d_partial, h->d_counter, beta + i, S + S_TMP + 4); }
    TDVP_TRY(lc(h, "k_lanczos_update"));
    { ProfScope _ps(st, "vec.k_scale_dev"); k_scale_dev<<<nb, RED_THREADS, 0, st>>>(w, w, N, beta + i, 0, 0.0); }
    TDVP_TRY(lc(h, "k_scale_dev"));
    const int k = (int)i + 1;
    { ProfScope _ps(st, "vec.k_tridiag_eigvec"); k_tridiag_eigvec<<<1, 32, 0, st>>>(k, alpha, beta, root, coef, work); }
    TDVP_TRY(lc(h, "k_tridiag_eigvec"));
    c128* y = ybuf[cur];
    { ProfScope _ps(st, "vec.k_combine_big");
      k_combine_big<<<nb, RED_THREADS, 0, st>>>(V, N, k, coef, y, have_prev ? ybuf[cur ^ 1] : nullptr, N, h->d_partial,
                                                  h->d_counter, S + S_ERR, S + S_YNORM); }
    TDVP_TRY(lc(h, "k_combine_big"));
    TDVP_CUDA(h, cudaMemcpyAsync(h->h_scal + S_BETA, beta + i, sizeof(double), cudaMemcpyDeviceToHost, st));
    TDVP_CUDA(h, cudaMemcpyAsync(h->h_scal + S_ERR, S + S_ERR, sizeof(double), cudaMemcpyDeviceToHost, st));
    TDVP_CUDA(h, cudaStreamSynchronize(st));
    const double b = h->h_scal[S_BETA];
    if (!(b == b)) { set_error(h, "lanczos_eigvec: NaN in the recurrence"); return TDVP_ERR_NOT_CONVERGED; }
    bool done = b < EPS_K;
    if (!done && i > 0) done = (h->h_scal[S_ERR] < thresh) || (i == N);
    if (!done && i == klimit) {
      // the reference raises here as well (3000 vectors); a memory-capped basis must not return an unconverged vector either
      set_error(h, klimit >= 3000 ? "Lanczos Diagonalization is not converged in 3000 basis"
                                  : "Lanczos Diagonalization is not converged: the Krylov basis hit the device-memory cap before 3000 vectors");
      return TDVP_ERR_NOT_CONVERGED;
    }
    if (done) {
      { ProfScope _ps(st, "vec.k_scale_dev"); k_scale_dev<<<nb, RED_THREADS, 0, st>>>(y, psi, N, S + S_YNORM, 0, 0.0); }
      TDVP_TRY(lc(h, "k_scale_dev"));
      if (niter) *niter = (int)i + 1;
      return 0;
    }
    have_prev = true;
    cur ^= 1;
  }
  set_error(h, "Lanczos Diagonalization is not converged in 3000 basis");
  return TDVP_ERR_NOT_CONVERGED;
}

}  // namespace tdvp
