// One C entry point around the library's own tdvp::gemm for tests/test_gpu_gemm_paths.py (loaded through ctypes, linked
// against the libtdvp_b200.so the Engine has loaded).  It runs any GemmDesc the contractions could build -- two-level
// rows, column-major C, conjugated operands -- and reports the plan plan_gemm made for it under the handle's context
// (the overrides of tdvp_set_gemm_config included), so a test can tell which kernel, reduction and tensor-map geometry
// it asked for.
#include "contract.cuh"
#include "zgemm_plan.h"

using namespace tdvp;

extern "C" {

// desc: M, N, K, A, a_m_inner, a_m1, a_m0, a_k, a_conj, B, b_n_inner, b_n1, b_n0, b_k, b_conj, C, c_m_inner, c_m1, c_m0,
//       c_n (pointers as addresses, strides in complex128 elements)
// ab:   alpha (re, im), beta (re, im)
// plan: kernel, S, k_chunk, reduce, c_stream, tiles_m, tiles_n, group_m, streamk, sk_tiles, grid, a_kmajor, b_kmajor,
//       a.small_inner, a.swapped, b.small_inner, b.swapped
// Returns the return code of tdvp::gemm (0, or the CUDA error of the launch).
int gemm_desc_run(void* handle, const long long* desc, const double* ab, long long* plan) {
  Handle* h = reinterpret_cast<Handle*>(handle);
  GemmDesc d;
  d.M = (int)desc[0]; d.N = (int)desc[1]; d.K = (int)desc[2];
  d.A = reinterpret_cast<const c128*>((uintptr_t)desc[3]);
  d.a_m_inner = (int)desc[4]; d.a_m1 = desc[5]; d.a_m0 = desc[6]; d.a_k = desc[7]; d.a_conj = (int)desc[8];
  d.B = reinterpret_cast<const c128*>((uintptr_t)desc[9]);
  d.b_n_inner = (int)desc[10]; d.b_n1 = desc[11]; d.b_n0 = desc[12]; d.b_k = desc[13]; d.b_conj = (int)desc[14];
  d.C = reinterpret_cast<c128*>((uintptr_t)desc[15]);
  d.c_m_inner = (int)desc[16]; d.c_m1 = desc[17]; d.c_m0 = desc[18]; d.c_n = desc[19];
  d.alpha = {ab[0], ab[1]};
  d.beta = {ab[2], ab[3]};
  d.tag = "test.gemm_desc";
  const GemmPlan p = plan_gemm(d, h->gemm);
  const long long v[17] = {p.kernel, p.S, p.k_chunk, p.reduce, p.c_stream, p.tiles_m, p.tiles_n, p.group_m, p.streamk,
                           p.sk_tiles, p.grid, p.a_kmajor, p.b_kmajor, p.a.small_inner, p.a.swapped, p.b.small_inner,
                           p.b.swapped};
  for (int i = 0; i < 17; ++i) plan[i] = v[i];
  return gemm(h, d, "gemm_desc_run");
}

}  // extern "C"
