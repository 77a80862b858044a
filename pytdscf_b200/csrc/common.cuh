// Shared declarations of libtdvp_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>
#include <cstdio>
#include <string>

namespace tdvp {

typedef double2 c128;  // complex128, interleaved (re, im): what NumPy / torch hold

// ---- error plumbing: every entry point returns int, never throws (include/tdvp_b200.h) -------
enum : int {
  TDVP_OK = 0,
  TDVP_ERR_ARG = -1,
  TDVP_ERR_SHAPE = -2,
  TDVP_ERR_NOT_CONVERGED = -3,
  TDVP_ERR_UNSUPPORTED = -4,
  TDVP_ERR_ZERO_NORM = -5,
};

struct Handle;
void set_error(Handle* h, const std::string& msg);
int cuda_fail(Handle* h, cudaError_t e, const char* what, const char* file, int line);

#define TDVP_CUDA(h, expr)                                              \
  do {                                                                  \
    cudaError_t _e = (expr);                                            \
    if (_e != cudaSuccess) return tdvp::cuda_fail((h), _e, #expr, __FILE__, __LINE__); \
  } while (0)

#define TDVP_TRY(expr)            \
  do {                            \
    int _rc = (expr);             \
    if (_rc != 0) return _rc;     \
  } while (0)

// ---- generalised GEMM descriptor -------------------------------------------------------------
// C[m,n] = alpha * sum_k opA[m,k] * opB[k,n] + beta * C[m,n], batched.
// Row / column indices may be two-level (m = m1*m_inner + m0) so that tensor contractions run on
// their natural layouts without transposes.  All strides are in complex128 elements.
struct GemmDesc {
  int M = 0, N = 0, K = 0, batch = 1;
  const c128* A = nullptr;
  long long a_batch = 0;   // batch stride
  int a_m_inner = 1;       // m = m1 * a_m_inner + m0
  long long a_m1 = 0, a_m0 = 0, a_k = 0;
  int a_conj = 0;          // use conj(A[m,k])
  const c128* B = nullptr;
  long long b_batch = 0;
  int b_n_inner = 1;
  long long b_n1 = 0, b_n0 = 0, b_k = 0;
  int b_conj = 0;
  c128* C = nullptr;
  long long c_batch = 0;
  int c_m_inner = 1;
  long long c_m1 = 0, c_m0 = 0, c_n = 1;
  c128 alpha = {1.0, 0.0};
  c128 beta = {0.0, 0.0};
  const char* tag = "gemm";   // profiling label (static string)
  // split-K (set by zgemm_auto): blockIdx.z = batch * splitk + split; split s covers k in [s*k_chunk, (s+1)*k_chunk)
  // and writes its partial to C + s * c_split (then combined by the fixed-order reduction kernel).
  int splitk = 1;
  int k_chunk = 0;
  long long c_split = 0;
  int c_stream = 0;   // set by the launcher: outputs larger than half of L2 are stored with evict-first (st.global.cs)
  // cluster split-K (tiny / small tiles, S <= 16): the S CTAs of a tile form a thread-block cluster along blockIdx.z; each
  // keeps its partial tile in its own shared memory and, after one cluster barrier, finishes 1/S of the tile by reading
  // the S partials through distributed shared memory in rank order.  C, alpha, beta are then the real ones (no scratch).
  int cluster_sk = 0;
};

// Per-handle (= per-device) launch context of the GEMM: stream, split-K scratch, device limits and the test /
// tuning overrides of tdvp_set_gemm_config (0 = automatic choice everywhere).
struct GemmCtx {
  cudaStream_t stream = nullptr;
  c128* scratch = nullptr;       // split-K partial products (may be null: no split-K)
  size_t scratch_elems = 0;
  int num_sms = 148;
  int force_cfg = 0;             // 1 big (128x64), 2 small (64x32), 3 tiny (32x32), 4 tma (persistent TMA-fed 128x64), 5 tma without stream-K
  int force_splitk = 0;          // 1 = never split, S >= 2 = S chunks (where K and the scratch allow it)
  int force_cstream = 0;         // 1 = evict-first stores of C always, 2 = never
  // stream-K fix-up buffers of the TMA kernel (one 128 x 64 accumulator image and one flag per CTA) and the launch epoch
  c128* sk_ws = nullptr;
  int* sk_flags = nullptr;
  int sk_slots = 0;
  mutable int sk_epoch = 0;
  bool tma_encode = false;       // the driver offers cuTensorMapEncodeTiled (queried once per handle)
};
constexpr size_t STREAMK_TILE_ELEMS = 128 * 64;
// Per-device kernel attributes (dynamic shared memory limits) and ctx.tma_encode: called by tdvp_create for every new handle.
cudaError_t zgemm_configure_device(GemmCtx& ctx);
// GEMM with automatic kernel, tile and split-K choice (plan_gemm in zgemm_plan.h); split-K partial products meet in a
// thread-block cluster or in ctx.scratch and are combined in fixed order, so results stay deterministic.  Returns
// cudaGetLastError() of the launch.
cudaError_t zgemm_auto(const GemmDesc& d, const GemmCtx& ctx);
constexpr size_t SPLITK_SCRATCH_ELEMS = size_t(18) << 20;  // 288 MiB of partial products
// Number of kernel launches issued through this library since load (bench.py's gpu_launches claim).
void count_launch(unsigned long long n = 1);
unsigned long long launch_count();
// Per-launch CUDA-event timing (off by default; used by bench.py for the roofline and the per-kernel breakdown).
// Every launch site brackets its kernel with prof_begin/prof_end on the launching stream; totals are kept per label.
void prof_enable(bool on);
bool prof_enabled();
void prof_begin(cudaStream_t stream, const char* label, double flops, bool is_gemm);
void prof_end(cudaStream_t stream);
void prof_collect(bool reset);                         // resolve pending events into the per-label totals
void prof_gemm_totals(double* ms, double* flops, unsigned long long* launches);
size_t prof_json(char* out, size_t cap);               // {"label": {"ms":..,"flops":..,"launches":..}, ...}
struct ProfScope {
  cudaStream_t s; bool on;
  ProfScope(cudaStream_t stream, const char* label, double flops = 0.0, bool is_gemm = false) : s(stream), on(prof_enabled()) {
    if (on) prof_begin(s, label, flops, is_gemm);
  }
  ~ProfScope() { if (on) prof_end(s); }
};

// Plain row-major helpers
inline GemmDesc gemm_rowmajor(int M, int N, int K, const c128* A, long long lda, bool transA, bool conjA,
                              const c128* B, long long ldb, bool transB, c128* C, long long ldc,
                              c128 alpha = {1.0, 0.0}, c128 beta = {0.0, 0.0}) {
  GemmDesc g;
  g.M = M; g.N = N; g.K = K;
  g.A = A; g.a_m_inner = 1; g.a_m0 = 0;
  if (!transA) { g.a_m1 = lda; g.a_k = 1; } else { g.a_m1 = 1; g.a_k = lda; }
  g.a_conj = conjA ? 1 : 0;
  g.B = B; g.b_n_inner = 1; g.b_n0 = 0;
  if (!transB) { g.b_n1 = 1; g.b_k = ldb; } else { g.b_n1 = ldb; g.b_k = 1; }
  g.C = C; g.c_m_inner = 1; g.c_m1 = ldc; g.c_m0 = 0; g.c_n = 1;
  g.alpha = alpha; g.beta = beta;
  return g;
}

inline GemmDesc tagged(GemmDesc g, const char* tag) { g.tag = tag; return g; }

__host__ __device__ inline c128 cmul(c128 a, c128 b) { return {a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x}; }
__host__ __device__ inline c128 cadd(c128 a, c128 b) { return {a.x + b.x, a.y + b.y}; }
__host__ __device__ inline c128 cconj(c128 a) { return {a.x, -a.y}; }

}  // namespace tdvp
