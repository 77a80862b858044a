// C entry points around pytdscf_b200/csrc/zgemm_plan.h for tests/test_gemm_plan_cpu.py (loaded through ctypes).  Operand
// pointers are plain addresses (only their alignment matters to the planner); nothing here touches a GPU.
#include "zgemm_plan.h"

using namespace tdvp;

namespace {

// desc: M, N, K, batch, A address, a_m_inner, a_m1, a_m0, a_k, B address, b_n_inner, b_n1, b_n0, b_k
GemmDesc make_desc(const long long* v) {
  GemmDesc d;
  d.M = (int)v[0]; d.N = (int)v[1]; d.K = (int)v[2]; d.batch = (int)v[3];
  d.A = reinterpret_cast<const c128*>((uintptr_t)v[4]);
  d.a_m_inner = (int)v[5]; d.a_m1 = v[6]; d.a_m0 = v[7]; d.a_k = v[8];
  d.B = reinterpret_cast<const c128*>((uintptr_t)v[9]);
  d.b_n_inner = (int)v[10]; d.b_n1 = v[11]; d.b_n0 = v[12]; d.b_k = v[13];
  return d;
}

// ctx: scratch present, scratch_elems, num_sms, force_cfg, force_splitk, force_cstream, stream-K buffers present, sk_slots,
//      tma_encode
GemmCtx make_ctx(const long long* v) {
  GemmCtx c;
  c.scratch = v[0] ? reinterpret_cast<c128*>((uintptr_t)256) : nullptr;
  c.scratch_elems = (size_t)v[1];
  c.num_sms = (int)v[2];
  c.force_cfg = (int)v[3]; c.force_splitk = (int)v[4]; c.force_cstream = (int)v[5];
  c.sk_ws = v[6] ? reinterpret_cast<c128*>((uintptr_t)512) : nullptr;
  c.sk_flags = v[6] ? reinterpret_cast<int*>((uintptr_t)1024) : nullptr;
  c.sk_slots = (int)v[7];
  c.tma_encode = v[8] != 0;
  return c;
}

}  // namespace

extern "C" {

// out: kernel, S, k_chunk, reduce, c_stream, tiles_m, tiles_n, group_m, streamk, sk_tiles, grid
void gemm_plan(const long long* desc, const long long* ctx, long long* out) {
  const GemmPlan p = plan_gemm(make_desc(desc), make_ctx(ctx));
  const long long v[11] = {p.kernel, p.S, p.k_chunk, p.reduce, p.c_stream, p.tiles_m, p.tiles_n,
                           p.group_m, p.streamk, p.sk_tiles, p.grid};
  for (int i = 0; i < 11; ++i) out[i] = v[i];
}

// out: streamk, sk_tiles, grid of `total` single-split work items of KT k-tiles
void gemm_plan_streamk(long long total, int KT, const long long* ctx, long long* out) {
  GemmPlan p;
  plan_streamk(p, total, KT, make_ctx(ctx));
  out[0] = p.streamk; out[1] = p.sk_tiles; out[2] = p.grid;
}

// plan_side on one operand: 1 when a tensor map can describe it with R-row boxes
int gemm_plan_side_ok(long long addr, long long rows, int K, int inner, long long s1, long long s0, long long sk, int R) {
  SidePlan pl;
  TmaSide side;
  bool kmajor;
  return plan_side(&pl, &side, &kmajor, reinterpret_cast<const c128*>((uintptr_t)addr), rows, K, inner, s1, s0, sk, R) ? 1 : 0;
}

// Segments of CTA `cta` of `grid` in execution order (get_seg for si = 0 .. seg_count - 1), 6 ints each: tm, tn, split,
// kt0, kt1, role.  Returns the count; at most `cap` are written.
int gemm_plan_segments(int tiles_m, int tiles_n, int splitk, int K, int k_chunk, int group_m, int streamk, int sk_tiles, int cta,
                       int grid, int* out, int cap) {
  TmaParams p = {};
  p.tiles_m = tiles_m; p.tiles_n = tiles_n; p.splitk = splitk; p.K = K; p.k_chunk = k_chunk; p.group_m = group_m;
  p.streamk = streamk; p.sk_tiles = sk_tiles;
  const int KT = (K + TMA_BK - 1) / TMA_BK;
  const int n = seg_count(p, KT, cta, grid);
  for (int si = 0; si < n && si < cap; ++si) {
    const Seg s = get_seg(p, si, KT, cta, grid);
    const int v[6] = {s.tm, s.tn, s.split, s.kt0, s.kt1, s.role};
    for (int i = 0; i < 6; ++i) out[6 * si + i] = v[i];
  }
  return n;
}

}  // extern "C"
