// Launch plan of every ZGEMM (zgemm_auto): which kernel runs, the split-K factor and where the partial sums meet, the
// store policy of C and, for the persistent TMA kernel, the tensor-map geometry of both operands, the rasterisation group
// and the stream-K schedule.  Every override of tdvp_set_gemm_config is interpreted here and nowhere else.
//
// Host logic only (no CUDA runtime or driver call): the header compiles with a plain C++ compiler given the CUDA include
// directory, and tests/test_streamk_schedule_cpu.py checks plan_gemm and the stream-K work assignment through a small shim
// (tests/c/gemm_plan_shim.cpp).  The work assignment at the end is the code zgemm_tma_kernel runs.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace tdvp {

// ---- kernels (the cp.async values are the tile_cfg values of tdvp_set_gemm_config) -----------------------------------
enum GemmKernel : int {
  GEMM_BIG = 1,       // cp.async 128 x 64 (zgemm.cu)
  GEMM_SMALL = 2,     // cp.async  64 x 32
  GEMM_TINY = 3,      // cp.async  32 x 32
  GEMM_TMA_WIDE = 4,  // persistent TMA-fed 128 x 64 (zgemm_tma.cu)
  GEMM_TMA_TALL = 5,  // persistent TMA-fed 256 x 32
};
enum GemmReduce : int {
  REDUCE_NONE = 0,
  REDUCE_CLUSTER = 1,   // the S CTAs of a tile form a thread-block cluster and sum through distributed shared memory
  REDUCE_SCRATCH = 2,   // partials go to GemmCtx::scratch, k_splitk_reduce sums them in fixed order
};

// ---- TMA kernel geometry and parameters -------------------------------------------------------------------------------
constexpr int TMA_BK = 16;
constexpr unsigned BIG_INNER = 1u << 30;   // "plain" operand: a single row level
// Two tile geometries, both 8 consumer warps of 32 x 32: 4 x 2 warps (CTA tile 128 x 64, 4 stages) for the bulk of the work and
// 8 x 1 warps (256 x 32, 3 stages) for GEMMs whose N is at most 32 (H_eff stage 2 at d w <= 32: with a 64-wide tile half of
// every B fragment would be zero padding).
template <int WMW_, int WNW_, int STAGES_>
struct TmaCfg {
  static constexpr int WMW = WMW_, WNW = WNW_, STAGES = STAGES_;
  static constexpr int BM = 32 * WMW, BN = 32 * WNW;
  static constexpr int SLAB_A = BM * 128, SLAB_B = BN * 128;          // bytes of one 8-k slab of the A / B tile
  static constexpr int STAGE_BYTES = 2 * (SLAB_A + SLAB_B);            // two slabs (BK = 16) of both operands
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 256;  // + alignment slack + barriers
  static_assert(WMW * WNW == 8, "8 consumer warps");
};
using WideCfg = TmaCfg<4, 2, 4>;     // 128 x 64, 4 x 48 KiB
using TallCfg = TmaCfg<8, 1, 3>;     // 256 x 32, 3 x 72 KiB

struct TmaSide {
  unsigned inner;      // rows per step of the outer row index (BIG_INNER: plain matrix)
  short small_inner;   // inner < tile rows: the box spans several outer steps
  short swapped;       // k-contiguous operand whose two row levels are listed (outer, inner) in the tensor map so that its
                       // strides ascend (the box has extent 1 in the outer level, the shared-memory image is the same)
};

struct TmaParams {
  int M, N, K, tiles_m, tiles_n, splitk, k_chunk;
  int group_m;         // M-tiles walked per N-tile before moving on: the A rows of a group stay in L2 while B streams
  TmaSide a, b;
  unsigned a_conj, b_conj;
  c128* C;
  int c_m_inner;
  long long c_m1, c_m0, c_n, c_split;
  c128 alpha, beta;
  int c_stream;
  // stream-K (splitk == 1, at least one tile per CTA): the tiles x k-tiles iteration space is cut into gridDim.x equal
  // contiguous ranges; a tile that straddles two ranges is finished by the second CTA from the first one's partial sums
  int streamk;         // 0: whole tiles round-robin (and split-K work items)
  int sk_tiles;        // stream-K: tiles [0, sk_tiles) are cut evenly over the CTAs, the rest are whole waves
  int epoch;           // value the head writer stores into sk_flags[cta] (grows with every launch: no reset needed)
  int* sk_flags;       // one per CTA
  c128* sk_ws;         // one BM x BN accumulator image per CTA, in fragment order
};

// Tensor-map geometry of one operand (the arguments of cuTensorMapEncodeTiled)
struct SidePlan {
  cuuint64_t dims[4], strides[3];
  cuuint32_t box[4];
};

inline cuuint64_t clamp_stride(unsigned long long s) {
  const unsigned long long cap = (1ull << 40) - 16;
  return s < 16 ? 16 : (s > cap ? cap : s);
}

// One operand with `rows` rows (two-level: row = r1 * inner + r0) and K columns, element (row, k) at
// ptr + r1 * s1 + r0 * s0 + k * sk (complex128 units).  R = tile rows (BM for A, BN for B).  Returns false when the
// operand cannot be described (the cp.async kernels then run).
inline bool plan_side(SidePlan* pl, TmaSide* side, bool* kmajor, const c128* ptr, long long rows, int K, int inner, long long s1,
                      long long s0, long long sk, int R) {
  cuuint64_t* dims = pl->dims;
  cuuint64_t* strides = pl->strides;
  cuuint32_t* box = pl->box;
  if (rows <= 0 || K < TMA_BK) return false;
  if ((reinterpret_cast<uintptr_t>(ptr) & 15u) != 0) return false;
  if (inner <= 0) return false;
  const bool two = inner > 1 && inner < rows;
  if (!two) {           // single row level: fold it into (inner = 1, s1)
    if (inner > 1) { s1 = s0; }   // rows <= inner: only the r0 level is walked
    inner = 1;
  } else if (rows % inner != 0) {
    return false;
  }
  if (sk == 1) {
    *kmajor = true;
    if (!two) {
      dims[0] = 2ull * K; dims[1] = (cuuint64_t)rows; dims[2] = 1; dims[3] = 1;
      strides[0] = clamp_stride(16ull * s1);
      strides[1] = clamp_stride(strides[0] * (unsigned long long)rows);
      strides[2] = strides[1];
      box[0] = 16; box[1] = R; box[2] = 1; box[3] = 1;
      side->inner = BIG_INNER; side->small_inner = 0; side->swapped = 0;
      if (s1 < 1) return false;
    } else {
      if (inner % R != 0 && R % inner != 0) return false;
      if (s0 < 1 || s1 < 1) return false;
      const long long n1 = rows / inner;
      const bool small = inner < R;
      const bool swap = !small && s0 > s1;
      dims[0] = 2ull * K; dims[3] = 1;
      if (!swap) {
        dims[1] = (cuuint64_t)inner; dims[2] = (cuuint64_t)n1;
        strides[0] = clamp_stride(16ull * s0);
        strides[1] = clamp_stride(16ull * s1);
        strides[2] = clamp_stride(strides[1] * (unsigned long long)n1);
        box[0] = 16; box[1] = small ? inner : R; box[2] = small ? R / inner : 1; box[3] = 1;
      } else {
        dims[1] = (cuuint64_t)n1; dims[2] = (cuuint64_t)inner;
        strides[0] = clamp_stride(16ull * s1);
        strides[1] = clamp_stride(16ull * s0);
        strides[2] = clamp_stride(strides[1] * (unsigned long long)inner);
        box[0] = 16; box[1] = 1; box[2] = R; box[3] = 1;
      }
      side->inner = (unsigned)inner; side->small_inner = small ? 1 : 0; side->swapped = swap ? 1 : 0;
    }
  } else {
    *kmajor = false;
    if (sk < 8) return false;        // k stride must cover the 8-row (128-byte) inner box
    if (!two) {
      if (s1 != 1 || rows % 8 != 0) return false;
      dims[0] = 16; dims[1] = (cuuint64_t)K; dims[2] = (cuuint64_t)(rows / 8); dims[3] = 1;
      strides[0] = clamp_stride(16ull * sk);
      strides[1] = 128;
      strides[2] = clamp_stride(128ull * (unsigned long long)(rows / 8));
      box[0] = 16; box[1] = 8; box[2] = R / 8; box[3] = 1;
      side->inner = BIG_INNER; side->small_inner = 0; side->swapped = 0;
    } else {
      if (s0 != 1 || inner % 8 != 0) return false;
      if (inner % R != 0 && R % inner != 0) return false;
      dims[0] = 16; dims[1] = (cuuint64_t)K; dims[2] = (cuuint64_t)(inner / 8); dims[3] = (cuuint64_t)(rows / inner);
      strides[0] = clamp_stride(16ull * sk);
      strides[1] = 128;
      strides[2] = clamp_stride(16ull * s1);
      const bool small = inner < R;
      box[0] = 16; box[1] = 8; box[2] = (small ? inner : R) / 8; box[3] = small ? R / inner : 1;
      side->inner = (unsigned)inner; side->small_inner = small ? 1 : 0; side->swapped = 0;
      if (s1 < 1) return false;
    }
  }
  for (int i = 0; i < 3; ++i)
    if (strides[i] % 16 != 0) return false;
  return true;
}

// ---- the plan ---------------------------------------------------------------------------------------------------------
struct GemmPlan {
  int kernel = GEMM_BIG;
  int S = 1;                 // split-K factor: split s covers k in [s k_chunk, (s + 1) k_chunk)
  int k_chunk = 0;           // a multiple of the tile's BK
  int reduce = REDUCE_NONE;  // REDUCE_NONE exactly when S == 1
  int c_stream = 0;          // evict-first stores of C (S == 1 only)
  // TMA kernels only.  Should the driver reject a tensor map the planner accepted, the cp.async big kernel runs the same
  // S, k_chunk and reduction instead.
  SidePlan a_map, b_map;
  TmaSide a, b;
  bool a_kmajor = false, b_kmajor = false;
  int tiles_m = 0, tiles_n = 0, group_m = 0, streamk = 0, sk_tiles = 0, grid = 0;
};

// Cost model of one launch (measured constants, profiles/r1_zgemm_cfg_sweep.json): a CTA tile of configuration c costs
// `lone` seconds per unit of k when it has an SM to itself and `full` when `cps` of them share the SM; K0 = prologue +
// epilogue in units of k.  time = waves * (k_chunk + K0) * per_k  (+ the fixed-order reduction for split-K).
struct CfgModel { int id, bm, bn, bk, cps, min_chunk; double lone, full, K0; };
constexpr CfgModel GEMM_MODELS[4] = {
    {4, 128, 64, 16, 1, 128, 0.2606e-6, 0.2606e-6, 40.0},  // tma: persistent big tile (7.70 ms on 8192x4096x1024, 0.231 ms on
                                                           // 1280x2560x256: profiles/r2_zgemm_shapes_tma.jsonl); replaces "big"
                                                           // whenever tensor maps can describe the operands
    {1, 128, 64, 16, 1, 128, 0.282e-6, 0.282e-6, 32.0},   // big   (8.33 ms / 28 waves / 1056 k on 8192x4096x1024)
    {2, 64, 32, 8, 4, 64, 0.075e-6, 0.30e-6, 24.0},       // small (only when forced: never the best in the sweep)
    {3, 32, 32, 8, 4, 32, 0.040e-6, 0.140e-6, 16.0},      // tiny  (832 us / 10.9 waves / 528 k on 1536x4096x512)
};

// Persistent grid and stream-K schedule of a TMA plan with `total` work items (tiles x S) of KT k-tiles each.
inline void plan_streamk(GemmPlan& pl, long long total, int KT, const GemmCtx& ctx) {
  pl.grid = (int)(total < ctx.num_sms ? total : ctx.num_sms);
  // stream-K whenever whole tiles would leave a ragged last round -- or between half as many tiles as SMs and all of them:
  // the ranges are then shorter than a tile and a tile's sums pass from one CTA to the next (this replaces split-K + its
  // reduction kernel for these shapes).  The kernel handles chains of any length, but each link costs ~4 us (128 KB out,
  // fence, flag, 128 KB in), so with fewer tiles than that the chain loses to split-K (measured: 8 tiles x 80 k-tiles ->
  // 114 us against 47 us, profiles/r2_zgemm_shapes_auto_chain.jsonl) and is not used.  Short K (< 16 k-tiles: H_eff stage
  // 2) loses more to the fix-up than it gains; force_cfg 5 = TMA kernel with whole tiles only (A/B tests)
  pl.streamk = 0;
  pl.sk_tiles = (int)total;
  if (pl.S == 1 && ctx.force_cfg != 5 && ctx.sk_ws && ctx.sk_flags && KT >= 16 && ctx.num_sms <= ctx.sk_slots) {
    if (total >= ctx.num_sms) {
      // only when the ragged last wave costs more than 3 %: with many waves stream-K gains nothing measurable and its
      // k-shifted first waves cost L2 reuse (8192 x 4096 x 1024, 27.7 waves: 617 MB of DRAM reads with, 522 MB without)
      const long long waves = (total + ctx.num_sms - 1) / ctx.num_sms;
      pl.streamk = ((waves * ctx.num_sms - total) * 100 > 3 * waves * ctx.num_sms || ctx.force_cfg == 4) ? 1 : 0;
      if (total % ctx.num_sms == 0) pl.streamk = 0;
      pl.sk_tiles = (int)(total % ctx.num_sms) + (total >= 2 * ctx.num_sms ? ctx.num_sms : 0);   // one to two waves' worth
      if (total < 2 * ctx.num_sms) pl.sk_tiles = (int)total;
    } else {
      pl.sk_tiles = (int)total;
      if (2 * total >= ctx.num_sms && KT >= 32) { pl.streamk = 1; pl.grid = ctx.num_sms; }   // <= 2 links, >= 16 k-tiles each
      else if (ctx.force_cfg == 4) {                      // forced "tma": long chains too (ranges of >= 4 k-tiles), for the tests
        long long g = total * KT / 4;
        if (g > ctx.num_sms) g = ctx.num_sms;
        if (g > total) { pl.streamk = 1; pl.grid = (int)g; }
      }
    }
  }
}

// Plan of `d` (M, N, batch > 0; its split-K fields at their defaults) under the handle's context.
inline GemmPlan plan_gemm(const GemmDesc& d, const GemmCtx& ctx) {
  GemmPlan pl;
  // ---- can tensor maps describe both operands?  N <= 32 with enough rows to fill the machine with 256-row tiles: tall
  const bool tall = d.N <= 32 && d.M >= 256 * 148;
  const int tbm = tall ? TallCfg::BM : WideCfg::BM, tbn = tall ? TallCfg::BN : WideCfg::BN;
  const bool tma_ok = (ctx.force_cfg == 0 || ctx.force_cfg >= 4) && d.batch == 1 && d.K >= TMA_BK && ctx.tma_encode &&
                      plan_side(&pl.a_map, &pl.a, &pl.a_kmajor, d.A, d.M, d.K, d.a_m_inner, d.a_m1, d.a_m0, d.a_k, tbm) &&
                      plan_side(&pl.b_map, &pl.b, &pl.b_kmajor, d.B, d.N, d.K, d.b_n_inner, d.b_n1, d.b_n0, d.b_k, tbn);

  // split-K through a thread-block cluster: tiny and small tiles, clusters of up to 16 CTAs (the non-portable size sm_100
  // offers; allowed per kernel in configure_cfg), one batch; force_cstream = 1 (a test override) keeps the scratch +
  // reduction-kernel path reachable for the tests
  auto cluster_ok = [&](int cfg, int S) {
    return (cfg == GEMM_SMALL || cfg == GEMM_TINY) && S >= 2 && S <= 16 && d.batch == 1 && ctx.force_cstream != 1;
  };
  auto tiles_of = [&](int bm, int bn) { return (long long)((d.M + bm - 1) / bm) * ((d.N + bn - 1) / bn) * d.batch; };

  // ---- wave-aware choice of the tile configuration AND the split-K factor (cost model above)
  int cfg = GEMM_BIG;
  double best_t = 1e30;
  const bool allow_split = ctx.scratch != nullptr && ctx.force_splitk != 1;
  // force_cfg 4 / 5 (tma) share the big tile's geometry: the split-K factor is chosen as for the forced big configuration
  const int forced = ctx.force_cfg >= 4 ? 1 : (ctx.force_cfg >= 1 && ctx.force_cfg <= 3 ? ctx.force_cfg : 0);
  const double bw = 5.0e12;
  // >= 8 full waves of big tiles with a long K: wave quantisation is < 6 % and the big tiles need the least L2 traffic
  // per flop (short-K GEMMs such as H_eff stage 2 are prologue-bound and keep the free choice)
  const bool large = tiles_of(128, 64) >= 8 * 148 && d.K >= 512;
  for (const CfgModel& m : GEMM_MODELS) {
    if (m.id == 4 ? !tma_ok : (m.id == 1 && tma_ok)) continue;           // the TMA kernel stands in for the big tile
    const int mid = m.id == 4 ? 1 : m.id;                                 // ... and shares its geometry / forcing rules
    if (forced ? forced != mid : (mid == 2 || (large && mid != 1))) continue;
    const long long tiles = tiles_of(m.bm, m.bn);
    const int slots = 148 * m.cps;
    int max_s = 1;
    if (allow_split && d.batch == 1 && d.K >= 2 * m.min_chunk && (tiles < 8 * 148 || ctx.force_splitk >= 2)) {
      max_s = d.K / m.min_chunk < 16 ? d.K / m.min_chunk : 16;
    }
    // tdvp_set_gemm_config(splitk = S >= 2): exactly that factor when the shape allows it (tests of the split-K path)
    const int min_s = (ctx.force_splitk >= 2 && max_s >= 2) ? (ctx.force_splitk < max_s ? ctx.force_splitk : max_s) : 1;
    if (min_s > 1) max_s = min_s;
    for (int S = min_s; S <= max_s; ++S) {
      int chunk = (d.K + S - 1) / S;
      chunk = (chunk + m.bk - 1) / m.bk * m.bk;
      if ((d.K + chunk - 1) / chunk != S) continue;
      if (S > 1 && (size_t)S * d.M * d.N > ctx.scratch_elems) break;
      const long long units = tiles * S;
      double per_k = m.full;
      if (units <= 148) per_k = m.lone;
      else if (units < slots) per_k = m.lone * (double)((units + 147) / 148);
      // big tiles run in lock-step waves (1 CTA per SM); the 4-per-SM tiny CTAs are scheduled dynamically, which the
      // sweep fits as fractional waves + half a wave of tail
      double waves = (double)((units + slots - 1) / slots);
      if (m.id == 3 && units >= slots) waves = (double)units / slots + 0.5;
      // the TMA kernel cuts the tiles x k-tiles space evenly over the SMs (stream-K): fractional waves + the fix-up (with
      // half..all as many tiles as SMs a tile is shared by two CTAs, one ~4 us hand-over)
      double sk_extra = 0.0;
      if (m.id == 4 && S == 1 && ctx.force_cfg != 5 && ctx.sk_ws) {
        if (units >= slots && d.K >= 256) waves = (double)units / slots + 0.1;
        else if (2 * units >= slots && d.K >= 512) { waves = (double)units / slots; sk_extra = 4.0e-6; }
      }
      double t = waves * (chunk + m.K0) * per_k + sk_extra;
      // split-K pays a second launch; in the launch-bound small-D regime that launch costs a full ~9 us slot of the stream
      // (r2 c2 profile: 2300 reduction launches per step), elsewhere ~4 us
      // -- unless the S CTAs of a tile can be a cluster (tiny / small tiles, S <= 8): then the partials meet in
      // distributed shared memory inside the same launch (two cluster barriers, ~2 us)
      if (S > 1 && cluster_ok(mid, S)) t += 2.0e-6;
      else if (S > 1) t += (double)(S + 2) * d.M * d.N * 16.0 / bw + ((double)d.M * d.N * d.K < 5.0e7 ? 9.0e-6 : 4.0e-6);
      if (t < best_t * (S > 1 && cfg == mid ? 0.97 : 1.0)) { best_t = t; cfg = mid; pl.S = S; pl.k_chunk = chunk; }
    }
  }

  // ---- reduction and store policy: outputs larger than half of L2 are written with evict-first stores
  if (pl.S < 2) pl.c_stream = ctx.force_cstream ? (ctx.force_cstream == 1) : ((double)d.M * d.N * d.batch * 16.0 > 64.0e6);
  else pl.reduce = cluster_ok(cfg, pl.S) ? REDUCE_CLUSTER : REDUCE_SCRATCH;

  // ---- the big-tile work goes to the persistent TMA kernel whenever tensor maps can describe the operands
  pl.kernel = cfg;
  if (!(ctx.force_cfg >= 4 || (ctx.force_cfg == 0 && cfg == GEMM_BIG)) || !tma_ok) return pl;
  const int BM = tall ? TallCfg::BM : WideCfg::BM, BN = tall ? TallCfg::BN : WideCfg::BN;
  const long long total = (long long)((d.M + BM - 1) / BM) * ((d.N + BN - 1) / BN) * pl.S;
  if (total > (1ll << 30)) return pl;
  pl.kernel = tall ? GEMM_TMA_TALL : GEMM_TMA_WIDE;
  pl.tiles_m = (d.M + BM - 1) / BM;
  pl.tiles_n = (d.N + BN - 1) / BN;
  // group of M-tiles whose A rows (group_m * BM * K complex) take ~32 MB: they stay in L2 while the group walks the N-tiles,
  // so B is read once per group.  ncu sweep on 8192 x 4096 x 1024 (algorithmic reads 201 MB): 693 / 617 / 778 / 1738 MB of
  // DRAM reads for 16 / 32 / 48 / 64 MB groups -- the two L2 partitions duplicate lines that SMs of both dies read, so the
  // usable capacity for an operand shared by all CTAs is about half of the 126 MB
  {
    const double a_tile_bytes = (double)BM * (double)d.K * 16.0;
    int gm = (int)(32.0e6 / a_tile_bytes);
    pl.group_m = gm < 8 ? 8 : (gm > 64 ? 64 : gm);
  }
  plan_streamk(pl, total, (d.K + TMA_BK - 1) / TMA_BK, ctx);
  return pl;
}

// ---- stream-K work assignment of zgemm_tma_kernel (CTA cta = blockIdx.x of grid = gridDim.x) ------------------------------------------------
struct Seg {
  int tm, tn, split, kt0, kt1, role;   // role 0: whole tile (or split-K item), 1: head part -> publish, 2: tail part -> finish,
                                       // 3: middle part (ranges shorter than a tile) -> add the predecessor's sums, publish
};

// Work item w -> (tile_m, tile_n, split): splits outermost, then the grouped rasterisation of zgemm_dmma_kernel (group_m
// M-tiles per N-tile), so the CTAs of one persistent "wave" (consecutive w) share A rows / B columns in L2.
__host__ __device__ __forceinline__ void decode_work(const TmaParams& p, int w, int& tm, int& tn, int& split) {
  const int GROUP_M = p.group_m;
  const int per_split = p.tiles_m * p.tiles_n;
  split = w / per_split;
  const int pid = w - split * per_split;
  const int in_group = GROUP_M * p.tiles_n;
  const int first_m = (pid / in_group) * GROUP_M;
  const int gsz = (p.tiles_m - first_m) < GROUP_M ? (p.tiles_m - first_m) : GROUP_M;
  tm = first_m + (pid % in_group) % gsz;
  tn = (pid % in_group) / gsz;
}

// Number of segments of this CTA and the si-th of them.  Stream-K is applied to the FIRST p.sk_tiles tiles of the raster only
// (between one and two waves' worth, or everything when there are fewer tiles than that): their tiles x k-tiles space is cut
// into `grid` equal contiguous ranges.  The remaining tiles are whole waves and keep the strided persistent order
// (tile = sk_tiles + w * grid + cta), in which the CTAs of a wave share A rows / B columns in L2 -- cutting the WHOLE raster
// into per-CTA ranges would put every CTA into a different region of the matrix at any moment and defeat that reuse
// (measured: 11 GB of DRAM reads instead of 0.5 GB on 8192 x 4096 x 1024).
// Order inside the stream-K part: the trailing partial tile (the HEAD part of a tile the next CTA finishes) first, then the
// whole tiles, the leading partial tile (TAIL part, finished here from the previous CTA's partial) last -- so a finisher
// never waits for work its neighbour has not started with.
__host__ __device__ __forceinline__ int sk_seg_count(const TmaParams& p, int KT, unsigned cta, unsigned grid) {
  const long long I = (long long)p.sk_tiles * KT;
  const long long a = I * cta / grid, b = I * (cta + 1) / grid;
  if (b <= a) return 0;
  const int first = (int)(a / KT), last = (int)((b - 1) / KT);
  return last - first + 1;       // lead (partial or whole) + middle tiles + trail (partial or whole)
}
__host__ __device__ __forceinline__ int seg_count(const TmaParams& p, int KT, unsigned cta, unsigned grid) {
  const int total = p.tiles_m * p.tiles_n * p.splitk;
  if (!p.streamk) return (int)cta < total ? (total - (int)cta + (int)grid - 1) / (int)grid : 0;
  const int rest = total - p.sk_tiles;    // a multiple of grid
  return sk_seg_count(p, KT, cta, grid) + rest / (int)grid;
}

__host__ __device__ __forceinline__ Seg get_seg(const TmaParams& p, int si, int KT, unsigned cta, unsigned grid) {
  Seg sg;
  if (!p.streamk) {
    const int w = cta + si * grid;
    decode_work(p, w, sg.tm, sg.tn, sg.split);
    const int k_begin = sg.split * p.k_chunk;
    const int k_end = (p.splitk > 1 && k_begin + p.k_chunk < p.K) ? k_begin + p.k_chunk : p.K;
    sg.kt0 = 0;
    sg.kt1 = (k_end - k_begin + TMA_BK - 1) / TMA_BK;
    sg.role = 0;
    return sg;
  }
  const int n = sk_seg_count(p, KT, cta, grid);
  if (si >= n) {                             // whole waves after the stream-K part
    decode_work(p, p.sk_tiles + (si - n) * (int)grid + (int)cta, sg.tm, sg.tn, sg.split);
    sg.kt0 = 0; sg.kt1 = KT; sg.role = 0;
    return sg;
  }
  const long long I = (long long)p.sk_tiles * KT;
  const long long a = I * cta / grid, b = I * (cta + 1) / grid;
  const int first = (int)(a / KT), a_off = (int)(a % KT), last = (int)((b - 1) / KT), b_off = (int)(b - (long long)last * KT);
  int tile;
  if (first == last) {                       // the whole range lies in one tile
    tile = first; sg.kt0 = a_off; sg.kt1 = b_off;
    sg.role = (a_off == 0 && b_off == KT) ? 0 : (a_off == 0 ? 1 : (b_off == KT ? 2 : 3));
  } else {
    // order: [trail, middle..., lead]
    if (si == 0) { tile = last; sg.kt0 = 0; sg.kt1 = b_off; sg.role = b_off == KT ? 0 : 1; }
    else if (si == n - 1) { tile = first; sg.kt0 = a_off; sg.kt1 = KT; sg.role = a_off == 0 ? 0 : 2; }
    else { tile = first + si; sg.kt0 = 0; sg.kt1 = KT; sg.role = 0; }
  }
  decode_work(p, tile, sg.tm, sg.tn, sg.split);
  return sg;
}

// ---- launchers of a plan ------------------------------------------------------------------------------------------------
cudaError_t zgemm_tma_configure_device(GemmCtx& ctx);
// Encode the plan's two tensor maps and launch the TMA kernel on `d` (split-K fields resolved); the cp.async big kernel
// when the driver rejects a map.
cudaError_t zgemm_tma_launch(const GemmDesc& d, const GemmPlan& pl, const GemmCtx& ctx);
// cp.async kernel GEMM_BIG / GEMM_SMALL / GEMM_TINY on `d` (split-K fields resolved)
cudaError_t zgemm_dmma_launch(int kernel, const GemmDesc& d, cudaStream_t stream);

}  // namespace tdvp
