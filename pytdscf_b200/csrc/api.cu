// extern "C" entry points of libtdvp_b200 (see include/tdvp_b200.h for the contract of each call).
#include <cstring>

#include "contract.cuh"

namespace tdvp {

int krylov_expm_exec(Handle* h, int kind, double scale_re, double scale_im, double thresh, int n_warmup,
                     int conserve_norm, const tdvp_heff_term* hterms, const tdvp_keff_term* kterms, int nterms,
                     int Dl, int d, int Dr, c128* psi, int* niter);
int lanczos_eigvec_exec(Handle* h, const tdvp_heff_term* hterms, int nterms, int Dl, int d, int Dr, c128* psi, int root,
                        double thresh, int* niter);
int inner_exec(Handle* h, long long n, const c128* bra, const c128* ket, int conj, c128* host_out);
int qr_shift_exec(Handle* h, int gauge, int Dl, int d, int Dr, const c128* psi, c128* site, c128* sigma);
int absorb_exec(Handle* h, int gauge, int Dl, int d, int Dr, int k, const c128* sigma, const c128* site, c128* out);
int qr_configure(Handle* h);
int svd_configure(Handle* h);

void set_error(Handle* h, const std::string& msg) {
  if (h) h->err = msg;
}

int cuda_fail(Handle* h, cudaError_t e, const char* what, const char* file, int line) {
  char buf[512];
  snprintf(buf, sizeof(buf), "CUDA error %d (%s) in %s at %s:%d", (int)e, cudaGetErrorString(e), what, file, line);
  set_error(h, buf);
  return (int)e > 0 ? (int)e : 1;
}

int ws_reserve(Handle* h, size_t bytes) {
  h->ws_top = 0;
  if (bytes <= h->ws_bytes) return 0;
  // grow geometrically; the old buffer may still be in use by enqueued work -> drain the stream first
  size_t want = bytes + bytes / 4 + (size_t(1) << 20);
  TDVP_CUDA(h, cudaStreamSynchronize(h->stream));
  if (h->side) TDVP_CUDA(h, cudaStreamSynchronize(h->side));
  if (h->ws) TDVP_CUDA(h, cudaFree(h->ws));
  h->ws = nullptr;
  h->ws_bytes = 0;
  void* p = nullptr;
  TDVP_CUDA(h, cudaMalloc(&p, want));
  h->ws = (unsigned char*)p;
  h->ws_bytes = want;
  return 0;
}

int ws_grow_preserve(Handle* h, size_t bytes) {
  if (bytes <= h->ws_bytes) return 0;
  void* p = nullptr;
  TDVP_CUDA(h, cudaMalloc(&p, bytes));
  if (h->ws) {
    cudaError_t e = cudaMemcpyAsync(p, h->ws, h->ws_top, cudaMemcpyDeviceToDevice, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) { cudaFree(p); return cuda_fail(h, e, "ws_grow_preserve copy", __FILE__, __LINE__); }
    TDVP_CUDA(h, cudaFree(h->ws));
  }
  h->ws = (unsigned char*)p;
  h->ws_bytes = bytes;
  return 0;
}

void* ws_alloc(Handle* h, size_t bytes) {
  const size_t b = align256(bytes);
  if (h->ws_top + b > h->ws_bytes) return nullptr;
  void* p = h->ws + h->ws_top;
  h->ws_top += b;
  return p;
}

}  // namespace tdvp

using namespace tdvp;

struct tdvp_handle_s : public tdvp::Handle {};

#define H_CHECK(h)            \
  if (!(h)) return TDVP_ERR_ARG; \
  (h)->err.clear();

extern "C" {

int tdvp_abi_version(void) { return 2; }

unsigned long long tdvp_launch_count(void) { return tdvp::launch_count(); }

int tdvp_create(int device, void* cuda_stream, tdvp_handle_t* out) {
  if (!out) return TDVP_ERR_ARG;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0) return e != cudaSuccess ? (int)e : (int)cudaErrorNoDevice;
  if (device < 0 || device >= ndev) return TDVP_ERR_ARG;
  if ((e = cudaSetDevice(device)) != cudaSuccess) return (int)e;
  tdvp_handle_s* h = new tdvp_handle_s();
  h->device = device;
  h->stream = (cudaStream_t)cuda_stream;
  if ((e = cudaMalloc((void**)&h->d_scal, 4096 * sizeof(double))) != cudaSuccess) { delete h; return (int)e; }
  if ((e = cudaMallocHost((void**)&h->h_scal, 4096 * sizeof(double))) != cudaSuccess) { delete h; return (int)e; }
  if ((e = cudaMalloc((void**)&h->d_partial, 1024 * 64 * sizeof(double))) != cudaSuccess) { delete h; return (int)e; }
  if ((e = cudaMalloc((void**)&h->d_counter, 16 * sizeof(unsigned int))) != cudaSuccess) { delete h; return (int)e; }
  if ((e = cudaMalloc((void**)&h->d_splitk, tdvp::SPLITK_SCRATCH_ELEMS * sizeof(c128))) != cudaSuccess) { delete h; return (int)e; }
  if ((e = cudaMalloc((void**)&h->d_partial_side, 1024 * 64 * sizeof(double))) != cudaSuccess ||
      (e = cudaMalloc((void**)&h->d_counter_side, 16 * sizeof(unsigned int))) != cudaSuccess ||
      (e = cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&h->ev_main, cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&h->ev_side, cudaEventDisableTiming)) != cudaSuccess) { tdvp_destroy(h); return (int)e; }
  cudaMemsetAsync(h->d_counter, 0, 16 * sizeof(unsigned int), h->stream);
  cudaMemsetAsync(h->d_counter_side, 0, 16 * sizeof(unsigned int), h->stream);
  cudaMemsetAsync(h->d_scal, 0, 4096 * sizeof(double), h->stream);
  memset(h->h_scal, 0, 4096 * sizeof(double));
  // device limits and kernel attributes are per device: (re)applied for every handle, never cached per process
  cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device);
  h->gemm.stream = h->stream;
  h->gemm.scratch = h->d_splitk;
  h->gemm.scratch_elems = tdvp::SPLITK_SCRATCH_ELEMS;
  h->gemm.num_sms = h->num_sms;
  h->gemm.sk_slots = h->num_sms;
  if ((e = cudaMalloc((void**)&h->gemm.sk_ws, sizeof(c128) * tdvp::STREAMK_TILE_ELEMS * (size_t)h->num_sms)) != cudaSuccess ||
      (e = cudaMalloc((void**)&h->gemm.sk_flags, sizeof(int) * (size_t)h->num_sms)) != cudaSuccess) { tdvp_destroy(h); return (int)e; }
  cudaMemsetAsync(h->gemm.sk_flags, 0, sizeof(int) * (size_t)h->num_sms, h->stream);
  int rc = 0;
  if ((e = tdvp::zgemm_configure_device(h->gemm)) != cudaSuccess) rc = (int)e;
  if (!rc) rc = tdvp::qr_configure(h);
  if (!rc) rc = tdvp::svd_configure(h);
  if (rc) { tdvp_destroy(h); return rc; }
  *out = h;
  return 0;
}

int tdvp_set_gemm_config(tdvp_handle_t h, int tile_cfg, int splitk, int c_stream) {
  if (!h || tile_cfg < 0 || tile_cfg > 5 || splitk < 0 || splitk > 16 || c_stream < 0 || c_stream > 2) return TDVP_ERR_ARG;
  h->gemm.force_cfg = tile_cfg;
  h->gemm.force_splitk = splitk;
  h->gemm.force_cstream = c_stream;
  return 0;
}

int tdvp_destroy(tdvp_handle_t h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  if (h->ws) cudaFree(h->ws);
  if (h->d_scal) cudaFree(h->d_scal);
  if (h->h_scal) cudaFreeHost(h->h_scal);
  if (h->d_partial) cudaFree(h->d_partial);
  if (h->d_counter) cudaFree(h->d_counter);
  if (h->d_splitk) cudaFree(h->d_splitk);
  if (h->side) { cudaStreamSynchronize(h->side); cudaStreamDestroy(h->side); }
  if (h->ev_main) cudaEventDestroy(h->ev_main);
  if (h->ev_side) cudaEventDestroy(h->ev_side);
  if (h->d_partial_side) cudaFree(h->d_partial_side);
  if (h->d_counter_side) cudaFree(h->d_counter_side);
  if (h->gemm.sk_ws) cudaFree(h->gemm.sk_ws);
  if (h->gemm.sk_flags) cudaFree(h->gemm.sk_flags);
  delete h;
  return 0;
}

const char* tdvp_last_error(tdvp_handle_t h) { return h ? h->err.c_str() : "null handle"; }

int tdvp_get_stats(tdvp_handle_t h, unsigned long long* solves, unsigned long long* matvecs, double* flops) {
  if (!h) return TDVP_ERR_ARG;
  if (solves) *solves = h->krylov_solves;
  if (matvecs) *matvecs = h->krylov_matvecs;
  if (flops) *flops = h->heff_flops;
  return 0;
}

int tdvp_reset_stats(tdvp_handle_t h) {
  if (!h) return TDVP_ERR_ARG;
  h->krylov_solves = 0;
  h->krylov_matvecs = 0;
  h->heff_flops = 0.0;
  return 0;
}

int tdvp_gemm_profile(int enable, int reset, double* ms, double* flops, unsigned long long* launches) {
  tdvp::prof_collect(false);
  tdvp::prof_gemm_totals(ms, flops, launches);
  if (reset) tdvp::prof_collect(true);
  tdvp::prof_enable(enable != 0);
  return 0;
}

size_t tdvp_profile_json(char* out, size_t cap) {
  tdvp::prof_collect(false);
  return tdvp::prof_json(out, cap);
}

int tdvp_heff_apply(tdvp_handle_t h, const tdvp_heff_term* terms, int nterms, int Dl, int d, int Dr,
                    const tdvp_c128* psi, tdvp_c128* out) {
  H_CHECK(h);
  if (!terms || !psi || !out || Dl <= 0 || d <= 0 || Dr <= 0) { set_error(h, "heff_apply: bad argument"); return TDVP_ERR_ARG; }
  if (psi == out) { set_error(h, "heff_apply: out must not alias psi"); return TDVP_ERR_ARG; }
  TDVP_TRY(ws_reserve(h, sizeof(c128) * heff_ws_elems(terms, nterms, Dl, d, Dr)));
  return heff_apply_exec(h, terms, nterms, Dl, d, Dr, (const c128*)psi, (c128*)out);
}

int tdvp_keff_apply(tdvp_handle_t h, const tdvp_keff_term* terms, int nterms, int Dl, int Dr, const tdvp_c128* sigma,
                    tdvp_c128* out) {
  H_CHECK(h);
  if (!terms || !sigma || !out || Dl <= 0 || Dr <= 0) { set_error(h, "keff_apply: bad argument"); return TDVP_ERR_ARG; }
  if (sigma == out) { set_error(h, "keff_apply: out must not alias sigma"); return TDVP_ERR_ARG; }
  TDVP_TRY(ws_reserve(h, sizeof(c128) * keff_ws_elems(terms, nterms, Dl, Dr)));
  return keff_apply_exec(h, terms, nterms, Dl, Dr, (const c128*)sigma, (c128*)out);
}

int tdvp_env_update(tdvp_handle_t h, int gauge, int Dl, int d, int Dr, const tdvp_c128* bra, const tdvp_c128* ket,
                    const tdvp_c128* E, int w_in, const tdvp_c128* W, int w_kind, int w_out, tdvp_c128* out,
                    int accumulate) {
  H_CHECK(h);
  if (!bra || !ket || !out || Dl <= 0 || d <= 0 || Dr <= 0 || w_in <= 0 || w_out <= 0) { set_error(h, "env_update: bad argument"); return TDVP_ERR_ARG; }
  TDVP_TRY(ws_reserve(h, sizeof(c128) * env_ws_elems(Dl, d, Dr, w_in, w_out)));
  return env_update_exec(h, gauge, Dl, d, Dr, (const c128*)bra, (const c128*)ket, (const c128*)E, w_in, (const c128*)W,
                         w_kind, w_out, (c128*)out, accumulate != 0);
}

int tdvp_set_krylov_size(tdvp_handle_t hh, long long size) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || size < 0) return TDVP_ERR_ARG;
  h->krylov_size_override = size;
  return 0;
}

int tdvp_krylov_expm(tdvp_handle_t h, int kind, double scale_re, double scale_im, double thresh, int n_warmup,
                     int conserve_norm, const tdvp_heff_term* hterms, const tdvp_keff_term* kterms, int nterms, int Dl,
                     int d, int Dr, tdvp_c128* psi_inout, int* niter) {
  H_CHECK(h);
  if (!psi_inout || nterms <= 0 || Dl <= 0 || Dr <= 0 || (hterms && d <= 0)) { set_error(h, "krylov_expm: bad argument"); return TDVP_ERR_ARG; }
  return krylov_expm_exec(h, kind, scale_re, scale_im, thresh, n_warmup, conserve_norm, hterms, kterms, nterms, Dl, d, Dr,
                          (c128*)psi_inout, niter);
}

int tdvp_lanczos_eigvec(tdvp_handle_t h, const tdvp_heff_term* hterms, int nterms, int Dl, int d, int Dr,
                        tdvp_c128* psi_inout, int root, double thresh, int* niter) {
  H_CHECK(h);
  if (!hterms || !psi_inout || nterms <= 0 || Dl <= 0 || d <= 0 || Dr <= 0) { set_error(h, "lanczos_eigvec: bad argument"); return TDVP_ERR_ARG; }
  return lanczos_eigvec_exec(h, hterms, nterms, Dl, d, Dr, (c128*)psi_inout, root, thresh, niter);
}

int tdvp_qr_shift(tdvp_handle_t h, int gauge, int Dl, int d, int Dr, const tdvp_c128* psi, tdvp_c128* site,
                  tdvp_c128* sigma) {
  H_CHECK(h);
  if (!psi || !site || !sigma || Dl <= 0 || d <= 0 || Dr <= 0) { set_error(h, "qr_shift: bad argument"); return TDVP_ERR_ARG; }
  return qr_shift_exec(h, gauge, Dl, d, Dr, (const c128*)psi, (c128*)site, (c128*)sigma);
}

int tdvp_absorb(tdvp_handle_t h, int gauge, int Dl, int d, int Dr, int k, const tdvp_c128* sigma, const tdvp_c128* site,
                tdvp_c128* out) {
  H_CHECK(h);
  if (!sigma || !site || !out || Dl <= 0 || d <= 0 || Dr <= 0 || k <= 0) { set_error(h, "absorb: bad argument"); return TDVP_ERR_ARG; }
  return absorb_exec(h, gauge, Dl, d, Dr, k, (const c128*)sigma, (const c128*)site, (c128*)out);
}

int tdvp_inner(tdvp_handle_t h, long long n, const tdvp_c128* bra, const tdvp_c128* ket, int conj, tdvp_c128* host_out) {
  H_CHECK(h);
  if (!bra || !ket || !host_out || n <= 0) { set_error(h, "inner: bad argument"); return TDVP_ERR_ARG; }
  return inner_exec(h, n, (const c128*)bra, (const c128*)ket, conj, (c128*)host_out);
}

int tdvp_overlap_site(tdvp_handle_t h, int Dlb, int Dlk, int d, int Drb, int Drk, const tdvp_c128* bra,
                      const tdvp_c128* ket, const tdvp_c128* block, int conj_bra, tdvp_c128* out) {
  H_CHECK(h);
  if (!bra || !ket || !block || !out) { set_error(h, "overlap_site: bad argument"); return TDVP_ERR_ARG; }
  TDVP_TRY(ws_reserve(h, sizeof(c128) * ((size_t)Dlb * d * Drk + 64)));
  return overlap_site_exec(h, Dlb, Dlk, d, Drb, Drk, (const c128*)bra, (const c128*)ket, (const c128*)block, conj_bra,
                           (c128*)out);
}

int tdvp_zgemm(tdvp_handle_t h, int transA, int transB, int M, int N, int K, double alpha_re, double alpha_im,
               const tdvp_c128* A, int lda, const tdvp_c128* B, int ldb, double beta_re, double beta_im, tdvp_c128* C,
               int ldc) {
  H_CHECK(h);
  if (!A || !B || !C || M < 0 || N < 0 || K < 0 || transA < 0 || transA > 2 || transB < 0 || transB > 2) {
    set_error(h, "zgemm: bad argument");
    return TDVP_ERR_ARG;
  }
  GemmDesc g = gemm_rowmajor(M, N, K, (const c128*)A, lda, transA != 0, transA == 2, (const c128*)B, ldb, transB != 0,
                             (c128*)C, ldc, c128{alpha_re, alpha_im}, c128{beta_re, beta_im});
  g.b_conj = transB == 2 ? 1 : 0;
  return gemm(h, g);
}

}  // extern "C"
