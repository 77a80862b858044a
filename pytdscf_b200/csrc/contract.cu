// H_eff / K_eff application and environment updates as chains of DMMA ZGEMMs on natural layouts.
//
// Replaces (reference file:line):
//   heff_term_exec   pytdscf/_contraction.py:1038-1176  (_op_lcr_dot, the (1|3, 1|3|4, 1|3) operand cases)
//   keff_term_exec   pytdscf/_contraction.py:1297-1352  (_op_lr_dot)
//   env_update_exec  pytdscf/_contraction.py:148-397    (contract_with_site_mpo)
//   overlap_site     pytdscf/wavefunction.py:248-255
//
// Contraction order is fixed to L -> W -> R (the minimum-flop order, SURVEY 8(d)):
//   T1[a,c,j,s] = sum_b L[a,c,b] psi[b,j,s]                 GEMM (Dl*wl) x (d*Dr) x Dl
//   T2[a,i,t,s] = sum_cj W[c,i,j,t] T1[a,c,j,s]              GEMM (Dl*Dr) x (d*wr) x (wl*d), two-level rows
//   out[a,i,r] += sum_ts T2[a,i,t,s] R[r,t,s]                GEMM (Dl*d) x Dr x (wr*Dr), B operand K-major
// The term sum is folded into the last GEMM's epilogue (beta = 1), so no separate accumulation pass.
#include "contract.cuh"

namespace tdvp {

namespace {

__global__ void permute_w_kernel(const c128* __restrict__ W, c128* __restrict__ Wp, int wl, int d, int wr, int mode) {
  // mode 0: Wp[c,j,i,t] = W[c,i,j,t]                 (W: wl,d,d,wr)
  // mode 1: Wp[q,s,r,p] = W[p,r,s,q]                 (W: wr',d,d,wl' with p=w_out, q=w_in; gauge-B mirror)
  const long long n = (long long)wl * d * d * wr;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < n; idx += (long long)gridDim.x * blockDim.x) {
    if (mode == 0) {
      int t = idx % wr; long long r = idx / wr;
      int i = r % d; r /= d;
      int j = r % d; int c = r / d;
      Wp[idx] = W[(((long long)c * d + i) * d + j) * wr + t];
    } else {
      // out index (q, s, r, p) with q in [0,wl) (=w_in), p in [0,wr) (=w_out); W is (p, r, s, q)
      int p = idx % wr; long long r_ = idx / wr;
      int r = r_ % d; r_ /= d;
      int s = r_ % d; int q = r_ / d;
      Wp[idx] = W[(((long long)p * d + r) * d + s) * wl + q];
    }
  }
}

__global__ void permute_wd_rev_kernel(const c128* __restrict__ W, c128* __restrict__ Wr, int wq, int d, int wp) {
  // Wr[q,r,p] = W[p,r,q]   (W: wp,d,wq)
  const long long n = (long long)wq * d * wp;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < n; idx += (long long)gridDim.x * blockDim.x) {
    int p = idx % wp; long long r_ = idx / wp;
    int r = r_ % d; int q = r_ / d;
    Wr[idx] = W[((long long)p * d + r) * wq + q];
  }
}

// out[r,j,l] = in[l,j,r]  (tiled transpose of the outer indices, one j-slab per blockIdx.z)
__global__ void permute_site_kernel(const c128* __restrict__ in, c128* __restrict__ out, int Dl, int d, int Dr) {
  __shared__ c128 tile[32][33];
  const int j = blockIdx.z;
  const int l0 = blockIdx.y * 32, r0 = blockIdx.x * 32;
  for (int y = threadIdx.y; y < 32; y += blockDim.y) {
    const int l = l0 + y, r = r0 + threadIdx.x;
    if (l < Dl && r < Dr) tile[y][threadIdx.x] = in[((long long)l * d + j) * Dr + r];
  }
  __syncthreads();
  for (int y = threadIdx.y; y < 32; y += blockDim.y) {
    const int r = r0 + y, l = l0 + threadIdx.x;
    if (l < Dl && r < Dr) out[((long long)r * d + j) * Dl + l] = tile[threadIdx.x][y];
  }
}

// T2[a,j,t,s] = alpha * sum_c Wd[c,j,t] * T1[a,c,j,s] + beta * T2[a,j,t,s]   (HBM-bound, s fastest)
__global__ void diag_mid_kernel(const c128* __restrict__ T1, const c128* __restrict__ Wd, c128* __restrict__ T2,
                                int Dl, int wl, int d, int wr, int Dr, c128 alpha, c128 beta) {
  extern __shared__ c128 wsm[];  // Wd[c, j, t] for this j: wl*wr entries
  const int j = blockIdx.y;
  const int a = blockIdx.z;
  for (int e = threadIdx.x; e < wl * wr; e += blockDim.x) {
    const int c = e / wr, t = e % wr;
    wsm[e] = Wd[((long long)c * d + j) * wr + t];
  }
  __syncthreads();
  const bool use_beta = beta.x != 0.0 || beta.y != 0.0;
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < Dr; s += gridDim.x * blockDim.x) {
    for (int t = 0; t < wr; ++t) {
      c128 acc = {0.0, 0.0};
      for (int c = 0; c < wl; ++c) {
        const c128 x = T1[(((long long)a * wl + c) * d + j) * Dr + s];
        const c128 w = wsm[c * wr + t];
        acc.x += w.x * x.x - w.y * x.y;
        acc.y += w.x * x.y + w.y * x.x;
      }
      c128* p = T2 + (((long long)a * d + j) * wr + t) * Dr + s;
      c128 o = cmul(alpha, acc);
      if (use_beta) o = cadd(o, cmul(beta, *p));
      *p = o;
    }
  }
}

__global__ void axpby_kernel(const c128* __restrict__ x, c128* __restrict__ y, long long n, c128 alpha, c128 beta) {
  const bool use_beta = beta.x != 0.0 || beta.y != 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    c128 o = cmul(alpha, x[i]);
    if (use_beta) o = cadd(o, cmul(beta, y[i]));
    y[i] = o;
  }
}

// y[r, c] = alpha * x[r, c] + beta * y[r, c] on row-strided 2-D views (cols contiguous)
__global__ void axpby2d_kernel(const c128* __restrict__ x, long long ldx, c128* __restrict__ y, long long ldy, long long rows,
                               int cols, c128 alpha, c128 beta) {
  const bool use_beta = beta.x != 0.0 || beta.y != 0.0;
  const long long tot = rows * cols;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x) {
    const long long r = e / cols;
    const int c = (int)(e % cols);
    c128 o = cmul(alpha, x[r * ldx + c]);
    c128* p = y + r * ldy + c;
    if (use_beta) o = cadd(o, cmul(beta, *p));
    *p = o;
  }
}

inline int grid_for(long long n, int threads, int cap = 148 * 8) {
  long long b = (n + threads - 1) / threads;
  if (b < 1) b = 1;
  if (b > cap) b = cap;
  return (int)b;
}

int launch_check(Handle* h, const char* what) {
  count_launch();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(h, e, what, __FILE__, __LINE__);
  return 0;
}

int axpby2d(Handle* h, const c128* x, long long ldx, c128* y, long long ldy, long long rows, int cols, c128 alpha, c128 beta) {
  { ProfScope _ps(h->stream, "aux.axpby2d_kernel"); axpby2d_kernel<<<grid_for(rows * cols, 256), 256, 0, h->stream>>>(x, ldx, y, ldy, rows, cols, alpha, beta); }
  return launch_check(h, "axpby2d_kernel");
}

// Identity-channel shortcuts pay only when the skipped GEMM slice is worth more than the extra copy / add launch.
constexpr long long ID_CHANNEL_MIN_ELEMS = 1ll << 17;

// C[(a, c), n] = sum_b L[(a, c), b] X[b, n] for every MPO channel c except `skip` (two-level rows over the remaining
// channels), and C[(a, skip), :] = X[a, :]  (L[:, skip, :] is the identity).
int left_apply_skip(Handle* h, const c128* L, int D, int w, int skip, const c128* X, long long ncols, c128* C, const char* tag) {
  int rc = 0;
  for (int part = 0; part < 2; ++part) {
    const int c0 = part == 0 ? 0 : skip + 1, c1 = part == 0 ? skip : w;
    if (c1 <= c0) continue;
    // GEMM rows ordered (channel outer, a inner): every 128-row tile then lies inside one channel, which is what lets the
    // TMA kernel describe L[:, c0:c1, :] and the matching rows of C with one box per tile
    GemmDesc g;
    g.M = D * (c1 - c0); g.N = (int)ncols; g.K = D;
    g.A = L + (long long)c0 * D; g.a_m_inner = D; g.a_m1 = D; g.a_m0 = (long long)w * D; g.a_k = 1;
    g.B = X; g.b_n_inner = 1; g.b_n1 = 1; g.b_n0 = 0; g.b_k = ncols;
    g.C = C + (long long)c0 * ncols; g.c_m_inner = D; g.c_m1 = ncols; g.c_m0 = (long long)w * ncols; g.c_n = 1;
    g.tag = tag;
    if ((rc = gemm(h, g))) return rc;
  }
  { ProfScope _ps(h->stream, "aux.id_channel_copy");
    cudaError_t e = cudaMemcpy2DAsync(C + (long long)skip * ncols, sizeof(c128) * (size_t)w * ncols, X, sizeof(c128) * (size_t)ncols,
                                      sizeof(c128) * (size_t)ncols, (size_t)D, cudaMemcpyDeviceToDevice, h->stream);
    if (e != cudaSuccess) return cuda_fail(h, e, "cudaMemcpy2DAsync(id channel)", __FILE__, __LINE__); }
  count_launch();
  return 0;
}

// out[m, r] = coef * sum_{(t, s), t != skip} T[m, (t, s)] R[r, (t, s)] + coef * T[m, skip, r] + beta * out[m, r]
// (R[:, skip, :] is the identity); T rows have w * Dr entries.
int right_apply_skip(Handle* h, const c128* T, long long rows, int Dr, int w, int skip, const c128* R, c128* out, c128 coef,
                     c128 beta_out, const char* tag) {
  int rc = 0;
  c128 beta = beta_out;
  const c128 one = {1.0, 0.0};
  for (int part = 0; part < 2; ++part) {
    const int t0 = part == 0 ? 0 : skip + 1, t1 = part == 0 ? skip : w;
    if (t1 <= t0) continue;
    GemmDesc g = gemm_rowmajor((int)rows, Dr, (t1 - t0) * Dr, T + (long long)t0 * Dr, (long long)w * Dr, false, false,
                               R + (long long)t0 * Dr, (long long)w * Dr, true, out, Dr, coef, beta);
    g.tag = tag;
    if ((rc = gemm(h, g))) return rc;
    beta = one;
  }
  return axpby2d(h, T + (long long)skip * Dr, (long long)w * Dr, out, Dr, rows, Dr, coef, beta);
}

int axpby(Handle* h, const c128* x, c128* y, long long n, c128 alpha, c128 beta) {
  { ProfScope _ps(h->stream, "aux.axpby_kernel"); axpby_kernel<<<grid_for(n, 256), 256, 0, h->stream>>>(x, y, n, alpha, beta); }
  return launch_check(h, "axpby_kernel");
}

// stage 2 with a full core: T2[a,i,t,s] = alpha * sum_{c,j} Wp[(c,j),(i,t)] T1[a,c,j,s] + beta*T2
int stage2_full(Handle* h, const c128* T1, const c128* Wp, c128* T2, int Dl, int wl, int d, int wr, int Dr,
                c128 alpha, c128 beta, const char* tag) {
  GemmDesc g;
  g.M = Dl * Dr; g.N = d * wr; g.K = wl * d;
  g.A = T1; g.a_m_inner = Dr; g.a_m1 = (long long)wl * d * Dr; g.a_m0 = 1; g.a_k = Dr;
  g.B = Wp; g.b_n_inner = 1; g.b_n1 = 1; g.b_n0 = 0; g.b_k = (long long)d * wr;
  g.C = T2; g.c_m_inner = Dr; g.c_m1 = (long long)d * wr * Dr; g.c_m0 = 1; g.c_n = Dr;
  g.alpha = alpha; g.beta = beta; g.tag = tag;
  return gemm(h, g);
}

int stage2_diag(Handle* h, const c128* T1, const c128* Wd, c128* T2, int Dl, int wl, int d, int wr, int Dr,
                c128 alpha, c128 beta) {
  const int threads = Dr >= 256 ? 256 : (Dr >= 128 ? 128 : (Dr >= 64 ? 64 : 32));
  dim3 grid((Dr + threads - 1) / threads, d, Dl);
  { ProfScope _ps(h->stream, "aux.diag_mid_kernel"); diag_mid_kernel<<<grid, threads, sizeof(c128) * wl * wr, h->stream>>>(T1, Wd, T2, Dl, wl, d, wr, Dr, alpha, beta); }
  return launch_check(h, "diag_mid_kernel");
}

}  // namespace

int gemm(Handle* h, const GemmDesc& g, const char* what) {
  cudaError_t e = zgemm_auto(g, h->gemm);
  if (e != cudaSuccess) return cuda_fail(h, e, what, __FILE__, __LINE__);
  return 0;
}

size_t heff_ws_elems(const tdvp_heff_term* terms, int nterms, int Dl, int d, int Dr) {
  size_t need = 0;
  for (int i = 0; i < nterms; ++i) {
    const tdvp_heff_term& t = terms[i];
    const size_t wl = t.L ? t.wl : 1, wr = t.R ? t.wr : 1;
    size_t e = (size_t)Dl * wl * d * Dr + (size_t)Dl * d * wr * Dr + (size_t)wl * d * d * wr + 64 * 3;
    if (e > need) need = e;
  }
  return need;
}

size_t keff_ws_elems(const tdvp_keff_term* terms, int nterms, int Dl, int Dr) {
  size_t need = 0;
  for (int i = 0; i < nterms; ++i) {
    const size_t w = (terms[i].L || terms[i].R) ? terms[i].w : 1;
    size_t e = (size_t)Dl * w * Dr + 64;
    if (e > need) need = e;
  }
  return need;
}

size_t env_ws_elems(int Dl, int d, int Dr, int w_in, int w_out) {
  const size_t D = Dl > Dr ? Dl : Dr;
  const size_t w = w_in > w_out ? w_in : w_out;
  return 2 * (size_t)Dl * d * Dr + 2 * D * D * d * w + (size_t)w_in * d * d * w_out + 64 * 6;
}

int heff_term_exec(Handle* h, const tdvp_heff_term& t, int Dl, int d, int Dr, const c128* psi, c128* out, bool accumulate) {
  const c128 coef = {t.coef_re, t.coef_im};
  const c128 one = {1.0, 0.0}, zero = {0.0, 0.0};
  const c128 beta_out = accumulate ? one : zero;
  const c128* L = reinterpret_cast<const c128*>(t.L);
  const c128* W = reinterpret_cast<const c128*>(t.W);
  const c128* R = reinterpret_cast<const c128*>(t.R);
  const int wl = L ? t.wl : 1, wr = R ? t.wr : 1;
  if (wl < 1 || wr < 1) { set_error(h, "heff term: MPO bond dimension < 1"); return TDVP_ERR_SHAPE; }
  if (!W && (wl != 1 || wr != 1)) {
    set_error(h, "heff term: identity core requires w_l == w_r == 1 (gap cores are unsupported, as in the reference)");
    return TDVP_ERR_UNSUPPORTED;
  }
  if (W && t.w_kind != TDVP_KIND_DIAG && t.w_kind != TDVP_KIND_FULL) { set_error(h, "heff term: bad w_kind"); return TDVP_ERR_ARG; }
  const int wlc = W ? t.wl : 1, wrc = W ? t.wr : 1;  // core bond dimensions
  if (W && ((L && wlc != wl) || (!L && wlc != 1) || (R && wrc != wr) || (!R && wrc != 1))) {
    set_error(h, "heff term: core bond dimensions do not match the environment blocks");
    return TDVP_ERR_SHAPE;
  }
  const size_t top = h->ws_top;
  const long long N = (long long)Dl * d * Dr;
  // identity channels promised by the caller (see tdvp_heff_term::id_channels); ignored for small tensors
  int l_id = (t.id_channels & 0xffff) - 1, r_id = ((t.id_channels >> 16) & 0xffff) - 1;
  if (N < ID_CHANNEL_MIN_ELEMS || !L || wl < 2 || l_id >= wl) l_id = -1;
  if (N < ID_CHANNEL_MIN_ELEMS || !R || wr < 2 || r_id >= wr) r_id = -1;
  // algorithmic flops (SURVEY 8(d))
  double fl = 0.0;
  if (L) fl += 8.0 * Dl * (double)Dl * Dr * d * wl;
  if (W) fl += (t.w_kind == TDVP_KIND_FULL ? 8.0 * Dl * (double)Dr * d * d * wl * wr : 8.0 * Dl * (double)Dr * d * wl * wr);
  if (R) fl += 8.0 * Dl * (double)Dr * Dr * d * wr;
  h->heff_flops += fl;

  const c128* cur = psi;
  int rc = 0;
  // ---- stage 1 ----
  if (L) {
    const bool last = !W && !R;
    c128* dst = last ? out : (c128*)ws_alloc(h, sizeof(c128) * (size_t)Dl * wl * d * Dr);
    if (!dst) { set_error(h, "workspace exhausted (heff T1)"); return TDVP_ERR_ARG; }
    if (l_id >= 0 && !last) {
      if ((rc = left_apply_skip(h, L, Dl, wl, l_id, cur, (long long)d * Dr, dst, "heff.s1"))) return rc;
    } else {
      GemmDesc g = gemm_rowmajor(Dl * wl, d * Dr, Dl, L, Dl, false, false, cur, (long long)d * Dr, false, dst,
                                 (long long)d * Dr, last ? coef : one, last ? beta_out : zero);
      g.tag = "heff.s1";
      if ((rc = gemm(h, g))) return rc;
    }
    cur = dst;
  }
  // ---- stage 2 ----
  if (W) {
    const bool last = !R;
    c128* dst = last ? out : (c128*)ws_alloc(h, sizeof(c128) * (size_t)Dl * d * wr * Dr);
    if (!dst) { set_error(h, "workspace exhausted (heff T2)"); return TDVP_ERR_ARG; }
    if (t.w_kind == TDVP_KIND_FULL) {
      const c128* Wp = reinterpret_cast<const c128*>(t.Wp);
      if (!Wp) {
        c128* tmp = (c128*)ws_alloc(h, sizeof(c128) * (size_t)wl * d * d * wr);
        if (!tmp) { set_error(h, "workspace exhausted (Wp)"); return TDVP_ERR_ARG; }
        { ProfScope _ps(h->stream, "aux.permute_w_kernel"); permute_w_kernel<<<grid_for((long long)wl * d * d * wr, 128, 64), 128, 0, h->stream>>>(W, tmp, wl, d, wr, 0); }
        if ((rc = launch_check(h, "permute_w_kernel"))) return rc;
        Wp = tmp;
      }
      rc = stage2_full(h, cur, Wp, dst, Dl, wl, d, wr, Dr, last ? coef : one, last ? beta_out : zero, "heff.s2");
    } else {
      rc = stage2_diag(h, cur, W, dst, Dl, wl, d, wr, Dr, last ? coef : one, last ? beta_out : zero);
    }
    if (rc) return rc;
    cur = dst;
  }
  // ---- stage 3 ----
  if (R) {
    if (r_id >= 0 && cur != psi) {
      if ((rc = right_apply_skip(h, cur, (long long)Dl * d, Dr, wr, r_id, R, out, coef, beta_out, "heff.s3"))) return rc;
    } else {
      GemmDesc g = gemm_rowmajor(Dl * d, Dr, wr * Dr, cur, (long long)wr * Dr, false, false, R, (long long)wr * Dr, true,
                                 out, Dr, coef, beta_out);
      g.tag = "heff.s3";
      if ((rc = gemm(h, g))) return rc;
    }
  } else if (!L && !W) {
    if ((rc = axpby(h, psi, out, N, coef, beta_out))) return rc;
  }
  h->ws_top = top;
  return 0;
}

int heff_apply_exec(Handle* h, const tdvp_heff_term* terms, int nterms, int Dl, int d, int Dr, const c128* psi, c128* out) {
  if (nterms <= 0) { set_error(h, "heff_apply: no terms"); return TDVP_ERR_ARG; }
  for (int i = 0; i < nterms; ++i) TDVP_TRY(heff_term_exec(h, terms[i], Dl, d, Dr, psi, out, i > 0));
  return 0;
}

int keff_term_exec(Handle* h, const tdvp_keff_term& t, int Dl, int Dr, const c128* sigma, c128* out, bool accumulate) {
  const c128 coef = {t.coef_re, t.coef_im};
  const c128 one = {1.0, 0.0}, zero = {0.0, 0.0};
  const c128 beta_out = accumulate ? one : zero;
  const c128* L = reinterpret_cast<const c128*>(t.L);
  const c128* R = reinterpret_cast<const c128*>(t.R);
  const int w = (L || R) ? t.w : 1;
  const size_t top = h->ws_top;
  int rc = 0;
  if (L && R) {
    h->heff_flops += 8.0 * w * ((double)Dl * Dl * Dr + (double)Dl * Dr * Dr);
    c128* T = (c128*)ws_alloc(h, sizeof(c128) * (size_t)Dl * w * Dr);
    if (!T) { set_error(h, "workspace exhausted (keff T)"); return TDVP_ERR_ARG; }
    int l_id = (t.id_channels & 0xffff) - 1, r_id = ((t.id_channels >> 16) & 0xffff) - 1;
    const bool big = (long long)Dl * Dr * w >= ID_CHANNEL_MIN_ELEMS && w >= 2;
    if (!big || l_id >= w) l_id = -1;
    if (!big || r_id >= w) r_id = -1;
    if (l_id >= 0) {
      if ((rc = left_apply_skip(h, L, Dl, w, l_id, sigma, Dr, T, "keff.g1"))) return rc;
    } else {
      GemmDesc g1 = gemm_rowmajor(Dl * w, Dr, Dl, L, Dl, false, false, sigma, Dr, false, T, Dr);
      g1.tag = "keff.g1";
      if ((rc = gemm(h, g1))) return rc;
    }
    if (r_id >= 0) {
      if ((rc = right_apply_skip(h, T, Dl, Dr, w, r_id, R, out, coef, beta_out, "keff.g2"))) return rc;
    } else {
      GemmDesc g2 = gemm_rowmajor(Dl, Dr, w * Dr, T, (long long)w * Dr, false, false, R, (long long)w * Dr, true, out, Dr, coef, beta_out);
      g2.tag = "keff.g2";
      if ((rc = gemm(h, g2))) return rc;
    }
  } else if (L || R) {
    if (w != 1) {
      set_error(h, "keff term: one-sided term requires w == 1");
      return TDVP_ERR_UNSUPPORTED;
    }
    if (L) {
      h->heff_flops += 8.0 * (double)Dl * Dl * Dr;
      GemmDesc g = tagged(gemm_rowmajor(Dl, Dr, Dl, L, Dl, false, false, sigma, Dr, false, out, Dr, coef, beta_out), "keff.one");
      if ((rc = gemm(h, g))) return rc;
    } else {
      h->heff_flops += 8.0 * (double)Dl * Dr * Dr;
      GemmDesc g = tagged(gemm_rowmajor(Dl, Dr, Dr, sigma, Dr, false, false, R, Dr, true, out, Dr, coef, beta_out), "keff.one");
      if ((rc = gemm(h, g))) return rc;
    }
  } else {
    if ((rc = axpby(h, sigma, out, (long long)Dl * Dr, coef, beta_out))) return rc;
  }
  h->ws_top = top;
  return 0;
}

int keff_apply_exec(Handle* h, const tdvp_keff_term* terms, int nterms, int Dl, int Dr, const c128* sigma, c128* out) {
  if (nterms <= 0) { set_error(h, "keff_apply: no terms"); return TDVP_ERR_ARG; }
  for (int i = 0; i < nterms; ++i) TDVP_TRY(keff_term_exec(h, terms[i], Dl, Dr, sigma, out, i > 0));
  return 0;
}

int permute_site(Handle* h, const c128* in, c128* out, int Dl, int d, int Dr) {
  dim3 grid((Dr + 31) / 32, (Dl + 31) / 32, d), block(32, 8);
  { ProfScope _ps(h->stream, "aux.permute_site_kernel"); permute_site_kernel<<<grid, block, 0, h->stream>>>(in, out, Dl, d, Dr); }
  return launch_check(h, "permute_site_kernel");
}

// gauge-A environment update on (possibly mirrored) operands:
//   out[i,q,j] (+)= sum conj(bra[m,r,i]) ket[n,s,j] E[m,p,n] W[p,r,s,q]
static int env_update_A(Handle* h, int Dl, int d, int Dr, const c128* bra, const c128* ket, const c128* E, int w_in,
                        const c128* W, const c128* Wp, int w_kind, int w_out, c128* out, bool accumulate) {
  const c128 one = {1.0, 0.0}, zero = {0.0, 0.0};
  int rc = 0;
  if (!W && (w_in != 1 || w_out != 1)) {
    set_error(h, "env_update: identity core requires w_in == w_out == 1");
    return TDVP_ERR_UNSUPPORTED;
  }
  if (!E && w_in != 1) { set_error(h, "env_update: identity block requires w_in == 1"); return TDVP_ERR_SHAPE; }
  double fl = 8.0 * Dl * (double)Dr * Dr * d * w_out;
  if (E) fl += 8.0 * Dl * (double)Dl * Dr * d * w_in;
  if (W) fl += (w_kind == TDVP_KIND_FULL ? 8.0 * Dl * (double)Dr * d * d * w_in * w_out : 8.0 * Dl * (double)Dr * d * w_in * w_out);
  h->heff_flops += fl;
  const c128* cur = ket;
  if (E) {
    c128* X = (c128*)ws_alloc(h, sizeof(c128) * (size_t)Dl * w_in * d * Dr);
    if (!X) { set_error(h, "workspace exhausted (env X)"); return TDVP_ERR_ARG; }
    GemmDesc g = tagged(gemm_rowmajor(Dl * w_in, d * Dr, Dl, E, Dl, false, false, ket, (long long)d * Dr, false, X, (long long)d * Dr), "env.s1");
    if ((rc = gemm(h, g))) return rc;
    cur = X;
  }
  if (W) {
    c128* Y = (c128*)ws_alloc(h, sizeof(c128) * (size_t)Dl * d * w_out * Dr);
    if (!Y) { set_error(h, "workspace exhausted (env Y)"); return TDVP_ERR_ARG; }
    if (w_kind == TDVP_KIND_FULL) rc = stage2_full(h, cur, Wp, Y, Dl, w_in, d, w_out, Dr, one, zero, "env.s2");
    else rc = stage2_diag(h, cur, W, Y, Dl, w_in, d, w_out, Dr, one, zero);
    if (rc) return rc;
    cur = Y;
  }
  // out[i,(q,j)] = sum_{(m,r)} conj(bra[(m,r), i]) * cur[(m,r),(q,j)]
  GemmDesc g = gemm_rowmajor(Dr, w_out * Dr, Dl * d, bra, Dr, true, true, cur, (long long)w_out * Dr, false, out,
                             (long long)w_out * Dr, one, accumulate ? one : zero);
  g.tag = "env.s3";
  return gemm(h, g);
}

int env_update_exec(Handle* h, int gauge, int Dl, int d, int Dr, const c128* bra, const c128* ket, const c128* E,
                    int w_in, const c128* W, int w_kind, int w_out, c128* out, bool accumulate) {
  const size_t top = h->ws_top;
  int rc = 0;
  if (W && w_kind != TDVP_KIND_DIAG && w_kind != TDVP_KIND_FULL) { set_error(h, "env_update: bad w_kind"); return TDVP_ERR_ARG; }
  if (gauge == TDVP_GAUGE_A) {
    const c128* Wp = nullptr;
    if (W && w_kind == TDVP_KIND_FULL) {
      c128* tmp = (c128*)ws_alloc(h, sizeof(c128) * (size_t)w_in * d * d * w_out);
      if (!tmp) { set_error(h, "workspace exhausted (env Wp)"); return TDVP_ERR_ARG; }
      { ProfScope _ps(h->stream, "aux.permute_w_kernel"); permute_w_kernel<<<grid_for((long long)w_in * d * d * w_out, 128, 64), 128, 0, h->stream>>>(W, tmp, w_in, d, w_out, 0); }
      if ((rc = launch_check(h, "permute_w_kernel"))) return rc;
      Wp = tmp;
    }
    rc = env_update_A(h, Dl, d, Dr, bra, ket, E, w_in, W, Wp, w_kind, w_out, out, accumulate);
  } else if (gauge == TDVP_GAUGE_B) {
    // mirror: Bt[m,r,i] = B[i,r,m]; E (Dr,w_in,Dr) plays the left block; W'[q,r,s,p] = W[p,r,s,q]
    c128* kt = (c128*)ws_alloc(h, sizeof(c128) * (size_t)Dl * d * Dr);
    if (!kt) { set_error(h, "workspace exhausted (env mirror)"); return TDVP_ERR_ARG; }
    if ((rc = permute_site(h, ket, kt, Dl, d, Dr))) return rc;
    c128* bt = kt;
    if (bra != ket) {
      bt = (c128*)ws_alloc(h, sizeof(c128) * (size_t)Dl * d * Dr);
      if (!bt) { set_error(h, "workspace exhausted (env mirror)"); return TDVP_ERR_ARG; }
      if ((rc = permute_site(h, bra, bt, Dl, d, Dr))) return rc;
    }
    const c128* Wm = nullptr;
    const c128* Wmp = nullptr;
    if (W) {
      c128* tmp = (c128*)ws_alloc(h, sizeof(c128) * (size_t)w_in * d * d * w_out);
      if (!tmp) { set_error(h, "workspace exhausted (env Wrev)"); return TDVP_ERR_ARG; }
      if (w_kind == TDVP_KIND_FULL) {
        { ProfScope _ps(h->stream, "aux.permute_w_kernel"); permute_w_kernel<<<grid_for((long long)w_in * d * d * w_out, 128, 64), 128, 0, h->stream>>>(W, tmp, w_in, d, w_out, 1); }
        if ((rc = launch_check(h, "permute_w_kernel"))) return rc;
        Wmp = tmp;
        Wm = tmp;  // only the permuted form is consumed for full cores
      } else {
        { ProfScope _ps(h->stream, "aux.permute_wd_rev_kernel"); permute_wd_rev_kernel<<<grid_for((long long)w_in * d * w_out, 128, 64), 128, 0, h->stream>>>(W, tmp, w_in, d, w_out); }
        if ((rc = launch_check(h, "permute_wd_rev_kernel"))) return rc;
        Wm = tmp;
      }
    }
    rc = env_update_A(h, Dr, d, Dl, bt, kt, E, w_in, Wm, Wmp, w_kind, w_out, out, accumulate);
  } else {
    set_error(h, "env_update: gauge must be TDVP_GAUGE_A or TDVP_GAUGE_B");
    return TDVP_ERR_ARG;
  }
  h->ws_top = top;
  return rc;
}

int overlap_site_exec(Handle* h, int Dlb, int Dlk, int d, int Drb, int Drk, const c128* bra, const c128* ket,
                      const c128* block, int conj_bra, c128* out) {
  const size_t top = h->ws_top;
  c128* X = (c128*)ws_alloc(h, sizeof(c128) * (size_t)Dlb * d * Drk);
  if (!X) { set_error(h, "workspace exhausted (overlap)"); return TDVP_ERR_ARG; }
  GemmDesc g1 = gemm_rowmajor(Dlb, d * Drk, Dlk, block, Dlk, false, false, ket, (long long)d * Drk, false, X, (long long)d * Drk);
  g1.tag = "ovlp.g1";
  TDVP_TRY(gemm(h, g1));
  GemmDesc g2 = gemm_rowmajor(Drb, Drk, Dlb * d, bra, Drb, true, conj_bra != 0, X, Drk, false, out, Drk);
  g2.tag = "ovlp.g2";
  TDVP_TRY(gemm(h, g2));
  h->ws_top = top;
  return 0;
}

}  // namespace tdvp
