// Complex128 GEMM on the FP64 tensor-core path of sm_100a (DMMA.8x8x4), the workhorse behind the
// H_eff / K_eff application, the environment updates, the bond absorb and the blocked QR.
//
// Replaces: opt_einsum.contract -> np.tensordot -> OpenBLAS ZGEMM in the reference
//           (pytdscf/_contraction.py:1162-1174, :1340-1352, :389-394; pytdscf/_mps_cls.py:1187-1206).
//
// Design notes (DESIGN.md "zgemm_dmma"):
//  * tcgen05/UMMA has no f64 kind; on sm_100a every mma.sync f64 shape lowers to DMMA.8x8x4
//    (cuobjdump of scripts/microbench/dmma_bench.cu), measured peak 37.0 TFLOP/s = 64 FMA/clk/SM
//    (profiles/r1_fp64_pipe_microbench.jsonl); cuBLAS ZGEMM 8192^3 reaches 36.97 TFLOP/s.
//  * complex product = 4 real DMMAs per (A-tile, B-tile) pair on fragments loaded as one LDS.128 per
//    complex element (re, im together), so HBM/L2/SMEM all keep the interleaved layout of the ABI.
//  * the FP64 pipe is ~30x slower than the SMEM crossbar needs, so the kernel is organised around
//    keeping 8 warps x 64 independent DMMAs in flight: CTA tile 128x64, warp tile 32x32, BK = 8,
//    4-stage cp.async (LDGSTS.128) ring, one __syncthreads per k-tile, XOR-swizzled SMEM so that
//    every fragment LDS.128 is bank-conflict free for both operand majors.
//  * rows of A/C and columns of B may be two-level indices (GemmDesc) so contractions such as
//    T2[a,i,t,s] = sum_{c,j} T1[a,c,j,s] W[c,i,j,t] run on their natural layouts (no transposes).
//  * round 2: this file keeps the cp.async kernels (three tile geometries), zgemm_auto and the two split-K forms --
//    scratch + fixed-order reduction kernel, and, for the small tiles, a thread-block cluster per output tile that reduces
//    the partial tiles through distributed shared memory.  The 128x64 work of the D >= 256 regime runs in the persistent
//    TMA-fed kernel of zgemm_tma.cu whenever tensor maps can describe the operands.  Which kernel, tile, split-K factor and
//    reduction a GEMM gets is decided by plan_gemm (zgemm_plan.h); zgemm_auto only executes the plan.
#include <cooperative_groups.h>

#include <atomic>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "zgemm_plan.h"

namespace tdvp {

namespace { std::atomic<unsigned long long> g_launches{0}; }
void count_launch(unsigned long long n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
unsigned long long launch_count() { return g_launches.load(std::memory_order_relaxed); }

// ---- optional per-launch timing (bench.py roofline / breakdown): CUDA events on the launching stream ----
namespace {
struct ProfTotals { double ms = 0.0, flops = 0.0; unsigned long long launches = 0; bool is_gemm = false; };
struct Pending { cudaEvent_t e0, e1; const char* label; };
struct Profiler {
  std::mutex mu;   // handles on several devices / host threads share the totals
  std::atomic<bool> enabled{false};
  std::vector<cudaEvent_t> pool;
  std::vector<Pending> pending;
  std::map<std::string, ProfTotals> totals;
  cudaEvent_t open_e0 = nullptr;
  const char* open_label = nullptr;
  cudaEvent_t get() {
    if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
  }
} g_prof;
}  // namespace

void prof_enable(bool on) { g_prof.enabled = on; }
bool prof_enabled() { return g_prof.enabled; }

// prof_begin .. prof_end bracket one launch and hold the lock in between (launch sites never nest)
void prof_begin(cudaStream_t stream, const char* label, double flops, bool is_gemm) {
  g_prof.mu.lock();
  ProfTotals& t = g_prof.totals[label];
  t.flops += flops;
  t.launches += 1;
  t.is_gemm = is_gemm;
  g_prof.open_e0 = g_prof.get();
  g_prof.open_label = label;
  cudaEventRecord(g_prof.open_e0, stream);
}

void prof_end(cudaStream_t stream) {
  cudaEvent_t e1 = g_prof.get();
  cudaEventRecord(e1, stream);
  g_prof.pending.push_back({g_prof.open_e0, e1, g_prof.open_label});
  g_prof.mu.unlock();
}

void prof_collect(bool reset) {
  std::lock_guard<std::mutex> lk(g_prof.mu);
  for (auto& pr : g_prof.pending) {
    cudaEventSynchronize(pr.e1);
    float t = 0.f;
    cudaEventElapsedTime(&t, pr.e0, pr.e1);
    g_prof.totals[pr.label].ms += t;
    g_prof.pool.push_back(pr.e0);
    g_prof.pool.push_back(pr.e1);
  }
  g_prof.pending.clear();
  if (reset) g_prof.totals.clear();
}

void prof_gemm_totals(double* ms, double* flops, unsigned long long* launches) {
  std::lock_guard<std::mutex> lk(g_prof.mu);
  double m = 0.0, f = 0.0;
  unsigned long long n = 0;
  for (auto& kv : g_prof.totals)
    if (kv.second.is_gemm) { m += kv.second.ms; f += kv.second.flops; n += kv.second.launches; }
  if (ms) *ms = m;
  if (flops) *flops = f;
  if (launches) *launches = n;
}

size_t prof_json(char* out, size_t cap) {
  std::lock_guard<std::mutex> lk(g_prof.mu);
  std::string js = "{";
  bool first = true;
  for (auto& kv : g_prof.totals) {
    char buf[256];
    snprintf(buf, sizeof(buf), "%s\"%s\": {\"ms\": %.6f, \"flops\": %.6e, \"launches\": %llu, \"gemm\": %s}", first ? "" : ", ",
             kv.first.c_str(), kv.second.ms, kv.second.flops, kv.second.launches, kv.second.is_gemm ? "true" : "false");
    js += buf;
    first = false;
  }
  js += "}";
  if (out && cap > 0) {
    size_t n = js.size() < cap - 1 ? js.size() : cap - 1;
    memcpy(out, js.data(), n);
    out[n] = 0;
  }
  return js.size() + 1;
}

namespace {

// Tile configurations.  Warp tile = (8 WI) x (8 WJ) complex, i.e. 4 WI WJ independent DMMA accumulations per k4-step.
//   Big:   4x2 warps of 32x32 -> CTA tile 128x64, BK = 16, 3 stages (144 KiB), 1 CTA/SM   (bulk of the D >= 256 work)
//   Small: 2x1 warps of 32x32 -> CTA tile  64x32, BK = 8,  4 stages ( 48 KiB), 4 CTAs/SM  (D <= 128: more CTAs, same 8 warps/SM)
//   Tiny:  2x2 warps of 16x16 -> CTA tile  32x32, BK = 8,  3 stages ( 24 KiB), 4+ CTAs/SM  (D <= 64: a warp reaches only its
//          SM sub-partition's quarter of the DMMA pipe, so latency-bound GEMMs want 4x less work per warp and 4x more warps)
template <int WMW_, int WNW_, int BK_, int STAGES_, int WI_ = 4, int WJ_ = 4>
struct Cfg {
  static constexpr int WMW = WMW_, WNW = WNW_, BK = BK_, STAGES = STAGES_, WI = WI_, WJ = WJ_;
  static constexpr int WTM = 8 * WI, WTN = 8 * WJ;
  static constexpr int BM = WTM * WMW, BN = WTN * WNW, THREADS = 32 * WMW * WNW;
  static constexpr int A_STAGE = BM * BK, B_STAGE = BN * BK;
  static constexpr int SMEM_BYTES = STAGES * (A_STAGE + B_STAGE) * (int)sizeof(c128);
  static constexpr int A_ITERS = A_STAGE / THREADS, B_ITERS = B_STAGE / THREADS;
  static_assert(THREADS % BK == 0 && THREADS % BM == 0 && THREADS % BN == 0, "tile / thread mapping");
};
using BigCfg = Cfg<4, 2, 16, 3>;
using SmallCfg = Cfg<2, 1, 8, 4>;
using TinyCfg = Cfg<2, 2, 8, 3, 2, 2>;

__device__ __forceinline__ void cp_async16(c128* smem, const c128* gmem, bool pred) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  int sz = pred ? 16 : 0;  // src-size 0 => zero fill, nothing is read
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

__device__ __forceinline__ double flip_sign(double x, unsigned mask) {
  return __hiloint2double(__double2hiint(x) ^ (int)mask, __double2loint(x));
}

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// SMEM chunk (16 B) index of tile element; the XOR keeps the 8 lanes of every LDS.128 phase on
// distinct 16-byte bank groups (see DESIGN.md for the bank arithmetic).
template <bool KMAJOR, int ROWS, int BK>
__device__ __forceinline__ int tile_chunk(int r, int k) {  // r: m or n inside the tile, k in [0, BK)
  if (KMAJOR) return r * BK + (k ^ ((r & 1) << 2));
  return k * ROWS + (r ^ ((k & 3) << 1));
}

// Per-thread global->shared copy plan of one operand tile (ROWS x BK), fixed for the whole k loop.
//   K-major (k contiguous in memory): thread owns k-chunk kc = tid % BK of rows tid / BK + (THREADS / BK) * i
//   row-major in m/n (the other index contiguous): thread owns row tid % ROWS for k = tid / ROWS + (THREADS / ROWS) * i
template <bool KMAJOR, int ROWS, int ITERS, int BK, int THREADS>
struct LoadPlan {
  long long off[KMAJOR ? ITERS : 1];
  unsigned ok;  // bit i: row of iteration i is inside the matrix
  __device__ __forceinline__ void init(int tid, int tile0, int extent, int inner, long long s1, long long s0) {
    ok = 0;
    if (KMAJOR) {
#pragma unroll
      for (int i = 0; i < ITERS; ++i) {
        const int r = tid / BK + (THREADS / BK) * i;
        const int m = tile0 + r;
        const bool in = m < extent;
        const int mm = in ? m : 0;
        off[i] = (long long)(mm / inner) * s1 + (long long)(mm % inner) * s0;
        ok |= (in ? 1u : 0u) << i;
      }
    } else {
      const int m = tile0 + tid % ROWS;
      const bool in = m < extent;
      const int mm = in ? m : 0;
      off[0] = (long long)(mm / inner) * s1 + (long long)(mm % inner) * s0;
      ok = in ? 0xffffffffu : 0u;
    }
  }
  __device__ __forceinline__ void issue(int tid, c128* smem, const c128* __restrict__ g, long long kstride, int k0, int k_end) const {
#pragma unroll
    for (int i = 0; i < ITERS; ++i) {
      int r, kl;
      long long o;
      if (KMAJOR) {
        r = tid / BK + (THREADS / BK) * i;
        kl = tid % BK;
        o = off[i];
      } else {
        r = tid % ROWS;
        kl = tid / ROWS + (THREADS / ROWS) * i;
        o = off[0];
      }
      const int k = k0 + kl;
      const bool p = ((ok >> i) & 1u) && (k < k_end);
      cp_async16(smem + tile_chunk<KMAJOR, ROWS, BK>(r, kl), p ? (g + o + (long long)k * kstride) : g, p);
    }
  }
};

template <typename C, bool A_KMAJOR, bool B_KMAJOR>
__global__ void __launch_bounds__(C::THREADS, C::THREADS == 256 ? 1 : 4) zgemm_dmma_kernel(const GemmDesc d) {
  constexpr int BM = C::BM, BN = C::BN, BK = C::BK, STAGES = C::STAGES, A_STAGE = C::A_STAGE, B_STAGE = C::B_STAGE;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  c128* As = reinterpret_cast<c128*>(smem_raw);
  c128* Bs = As + STAGES * A_STAGE;

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, q = lane & 3;
  const int wm = warp % C::WMW, wn = warp / C::WMW;
  // Grouped rasterisation: consecutive CTAs walk 16 M-tiles for one N-tile before moving to the next N-tile, so a wave of
  // 148 CTAs works on a 16 x ~9 block of tiles (A rows stay in L2 for the whole group, B columns are read once per
  // group) instead of ~2 full tile rows that stream all of B through L2 every wave.  blockIdx.x enumerates all tiles:
  // gridDim.y stops at 65535, which would cap M at 65535 tiles.
  int tile_m, tile_n;
  {
    constexpr int GROUP_M = 16;
    const int npm = (d.M + BM - 1) / BM, npn = (d.N + BN - 1) / BN;
    const int pid = blockIdx.x;
    const int in_group = GROUP_M * npn;
    const int first_m = (pid / in_group) * GROUP_M;
    const int gsz = (npm - first_m) < GROUP_M ? (npm - first_m) : GROUP_M;
    tile_m = (first_m + (pid % in_group) % gsz) * BM;
    tile_n = ((pid % in_group) / gsz) * BN;
  }
  const long long bz = blockIdx.z / d.splitk;
  const int split = blockIdx.z % d.splitk;
  const int k_begin = split * d.k_chunk;                       // k_chunk is a multiple of BK (or covers all of K)
  const int k_end = (d.splitk > 1 && k_begin + d.k_chunk < d.K) ? k_begin + d.k_chunk : d.K;
  const c128* __restrict__ Ag = d.A + bz * d.a_batch;
  const c128* __restrict__ Bg = d.B + bz * d.b_batch;
  c128* __restrict__ Cg = d.C + bz * d.c_batch + (long long)split * d.c_split;

  LoadPlan<A_KMAJOR, BM, C::A_ITERS, BK, C::THREADS> pa;
  LoadPlan<B_KMAJOR, BN, C::B_ITERS, BK, C::THREADS> pb;
  pa.init(tid, tile_m, d.M, d.a_m_inner, d.a_m1, d.a_m0);
  pb.init(tid, tile_n, d.N, d.b_n_inner, d.b_n1, d.b_n0);

  auto load_stage = [&](int stage, int k0) {
    pa.issue(tid, As + stage * A_STAGE, Ag, d.a_k, k0, k_end);
    pb.issue(tid, Bs + stage * B_STAGE, Bg, d.b_k, k0, k_end);
  };

  constexpr int WI = C::WI, WJ = C::WJ;
  double cre[WI][WJ][2], cim[WI][WJ][2];
#pragma unroll
  for (int i = 0; i < WI; ++i)
#pragma unroll
    for (int j = 0; j < WJ; ++j) {
      cre[i][j][0] = cre[i][j][1] = 0.0;
      cim[i][j][0] = cim[i][j][1] = 0.0;
    }

  const int KT = (k_end - k_begin + BK - 1) / BK;
#pragma unroll
  for (int s = 0; s < STAGES - 1; ++s) {
    if (s < KT) load_stage(s, k_begin + s * BK);
    cp_async_commit();
  }

  // conjugation / negation as integer sign-bit flips: keeps the FP64 pipe for the DMMAs only
  const unsigned sa = d.a_conj ? 0x80000000u : 0u;
  const unsigned sb = d.b_conj ? 0x80000000u : 0u;

  for (int kt = 0; kt < KT; ++kt) {
    cp_async_wait<STAGES - 2>();
    __syncthreads();
    {
      const int nk = kt + STAGES - 1;
      if (nk < KT) load_stage(nk % STAGES, k_begin + nk * BK);
      cp_async_commit();
    }
    const c128* as = As + (kt % STAGES) * A_STAGE;
    const c128* bs = Bs + (kt % STAGES) * B_STAGE;
#pragma unroll
    for (int k4 = 0; k4 < BK / 4; ++k4) {
      const int kk = k4 * 4 + q;
      double are[WI], aim[WI], naim[WI], bre[WJ], bim[WJ];
#pragma unroll
      for (int i = 0; i < WI; ++i) {
        const int r = wm * C::WTM + 8 * i + g;
        const c128 v = as[tile_chunk<A_KMAJOR, BM, BK>(r, kk)];
        are[i] = v.x;
        aim[i] = flip_sign(v.y, sa);
        naim[i] = flip_sign(v.y, sa ^ 0x80000000u);
      }
#pragma unroll
      for (int j = 0; j < WJ; ++j) {
        const int r = wn * C::WTN + 8 * j + g;
        const c128 v = bs[tile_chunk<B_KMAJOR, BN, BK>(r, kk)];
        bre[j] = v.x;
        bim[j] = flip_sign(v.y, sb);
      }
      // two passes so that dependent accumulations into the same tile are 2 WI WJ DMMAs apart
#pragma unroll
      for (int i = 0; i < WI; ++i)
#pragma unroll
        for (int j = 0; j < WJ; ++j) {
          dmma(cre[i][j][0], cre[i][j][1], are[i], bre[j]);
          dmma(cim[i][j][0], cim[i][j][1], are[i], bim[j]);
        }
#pragma unroll
      for (int i = 0; i < WI; ++i)
#pragma unroll
        for (int j = 0; j < WJ; ++j) {
          dmma(cre[i][j][0], cre[i][j][1], naim[i], bim[j]);
          dmma(cim[i][j][0], cim[i][j][1], aim[i], bre[j]);
        }
    }
  }
  cp_async_wait<0>();

  // ---- epilogue: C = alpha * acc + beta * C ----
  const c128 alpha = d.alpha, beta = d.beta;
  const bool use_beta = (beta.x != 0.0) || (beta.y != 0.0);
  if (d.cluster_sk) {
    // Cluster split-K: partial tiles meet in distributed shared memory instead of a scratch buffer + reduction launch.
    // Layout [register c = (i, j, e)][thread]: a warp reads 32 consecutive 16-byte words of the remote CTA.
    static_assert(WI * WJ * 2 * C::THREADS * (int)sizeof(c128) <= C::SMEM_BYTES, "partial tile must fit the stage buffers");
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __syncthreads();                                   // every warp is done with the stage buffers
    c128* part = reinterpret_cast<c128*>(smem_raw);
#pragma unroll
    for (int i = 0; i < WI; ++i)
#pragma unroll
      for (int j = 0; j < WJ; ++j)
#pragma unroll
        for (int e = 0; e < 2; ++e) part[((i * WJ + j) * 2 + e) * C::THREADS + tid] = c128{cre[i][j][e], cim[i][j][e]};
    cluster.sync();
    const int S = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
#pragma unroll
    for (int i = 0; i < WI; ++i) {
      const int m = tile_m + wm * C::WTM + 8 * i + g;
      const long long roff = (long long)(m / d.c_m_inner) * d.c_m1 + (long long)(m % d.c_m_inner) * d.c_m0;
#pragma unroll
      for (int j = 0; j < WJ; ++j) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int c = (i * WJ + j) * 2 + e;
          const int n = tile_n + wn * C::WTN + 8 * j + 2 * q + e;
          if (c % S != rank || m >= d.M || n >= d.N) continue;
          double sx = 0.0, sy = 0.0;
          for (int r = 0; r < S; ++r) {                // fixed order: rank 0 .. S-1 = ascending k
            const c128 v = cluster.map_shared_rank(part, r)[c * C::THREADS + tid];
            sx += v.x;
            sy += v.y;
          }
          c128* p = d.C + bz * d.c_batch + roff + (long long)n * d.c_n;
          c128 out = cmul(alpha, c128{sx, sy});
          if (use_beta) out = cadd(out, cmul(beta, *p));
          *p = out;
        }
      }
    }
    cluster.sync();                                    // nobody leaves while its partial may still be read
    return;
  }
#pragma unroll
  for (int i = 0; i < WI; ++i) {
    const int m = tile_m + wm * C::WTM + 8 * i + g;
    if (m >= d.M) continue;
    const long long roff = (long long)(m / d.c_m_inner) * d.c_m1 + (long long)(m % d.c_m_inner) * d.c_m0;
#pragma unroll
    for (int j = 0; j < WJ; ++j) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int n = tile_n + wn * C::WTN + 8 * j + 2 * q + e;
        if (n >= d.N) continue;
        c128* p = Cg + roff + (long long)n * d.c_n;
        c128 acc = {cre[i][j][e], cim[i][j][e]};
        c128 out = cmul(alpha, acc);
        if (use_beta) out = cadd(out, cmul(beta, *p));
        if (d.c_stream) __stcs(reinterpret_cast<double2*>(p), make_double2(out.x, out.y));
        else *p = out;
      }
    }
  }
}

template <typename C>
cudaError_t configure_cfg() {
  cudaError_t e;
  if (C::THREADS < 256) {   // tiny / small tiles: cluster split-K with up to 16 CTAs per tile
    if ((e = cudaFuncSetAttribute(zgemm_dmma_kernel<C, true, true>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1))) return e;
    if ((e = cudaFuncSetAttribute(zgemm_dmma_kernel<C, true, false>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1))) return e;
    if ((e = cudaFuncSetAttribute(zgemm_dmma_kernel<C, false, true>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1))) return e;
    if ((e = cudaFuncSetAttribute(zgemm_dmma_kernel<C, false, false>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1))) return e;
  }
  if ((e = cudaFuncSetAttribute(zgemm_dmma_kernel<C, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES))) return e;
  if ((e = cudaFuncSetAttribute(zgemm_dmma_kernel<C, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES))) return e;
  if ((e = cudaFuncSetAttribute(zgemm_dmma_kernel<C, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES))) return e;
  return cudaFuncSetAttribute(zgemm_dmma_kernel<C, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
}

template <typename C>
cudaError_t launch_cfg(const GemmDesc& d, cudaStream_t stream) {
  dim3 grid(((d.N + C::BN - 1) / C::BN) * ((d.M + C::BM - 1) / C::BM), 1, d.batch * d.splitk);
  const bool ak = (d.a_k == 1), bk = (d.b_k == 1);
  ProfScope scope(stream, d.tag, 8.0 * (double)d.M * (double)d.N * (double)d.K * (double)d.batch, true);
  if (d.cluster_sk) {
    cudaLaunchConfig_t lc = {};
    lc.gridDim = grid;
    lc.blockDim = dim3(C::THREADS);
    lc.dynamicSmemBytes = C::SMEM_BYTES;
    lc.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 1;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = (unsigned)d.splitk;
    lc.attrs = at;
    lc.numAttrs = 1;
    cudaError_t e;
    if (ak && bk) e = cudaLaunchKernelEx(&lc, zgemm_dmma_kernel<C, true, true>, d);
    else if (ak && !bk) e = cudaLaunchKernelEx(&lc, zgemm_dmma_kernel<C, true, false>, d);
    else if (!ak && bk) e = cudaLaunchKernelEx(&lc, zgemm_dmma_kernel<C, false, true>, d);
    else e = cudaLaunchKernelEx(&lc, zgemm_dmma_kernel<C, false, false>, d);
    count_launch();
    return e != cudaSuccess ? e : cudaGetLastError();
  }
  if (ak && bk)
    zgemm_dmma_kernel<C, true, true><<<grid, C::THREADS, C::SMEM_BYTES, stream>>>(d);
  else if (ak && !bk)
    zgemm_dmma_kernel<C, true, false><<<grid, C::THREADS, C::SMEM_BYTES, stream>>>(d);
  else if (!ak && bk)
    zgemm_dmma_kernel<C, false, true><<<grid, C::THREADS, C::SMEM_BYTES, stream>>>(d);
  else
    zgemm_dmma_kernel<C, false, false><<<grid, C::THREADS, C::SMEM_BYTES, stream>>>(d);
  count_launch();
  return cudaGetLastError();
}

}  // namespace

namespace {
// C[m,n] = alpha * sum_s P[s][m][n] + beta * C[m,n]   (fixed summation order over s; C addressed like GemmDesc)
__global__ void k_splitk_reduce(const c128* __restrict__ P, int S, int M, int N, long long stride, GemmDesc d) {
  const long long tot = (long long)M * N;
  const bool use_beta = d.beta.x != 0.0 || d.beta.y != 0.0;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x) {
    const int m = (int)(e / N), n = (int)(e % N);
    double sx = 0.0, sy = 0.0;
    for (int s = 0; s < S; ++s) {
      const c128 v = P[(long long)s * stride + e];
      sx += v.x;
      sy += v.y;
    }
    c128* p = d.C + (long long)(m / d.c_m_inner) * d.c_m1 + (long long)(m % d.c_m_inner) * d.c_m0 + (long long)n * d.c_n;
    c128 o = cmul(d.alpha, c128{sx, sy});
    if (use_beta) o = cadd(o, cmul(d.beta, *p));
    *p = o;
  }
}
}  // namespace

cudaError_t zgemm_dmma_launch(int kernel, const GemmDesc& d, cudaStream_t stream) {
  if (kernel == GEMM_TINY) return launch_cfg<TinyCfg>(d, stream);
  if (kernel == GEMM_SMALL) return launch_cfg<SmallCfg>(d, stream);
  return launch_cfg<BigCfg>(d, stream);
}

cudaError_t zgemm_configure_device(GemmCtx& ctx) {
  cudaError_t e;
  if ((e = zgemm_tma_configure_device(ctx))) return e;
  if ((e = configure_cfg<BigCfg>())) return e;
  if ((e = configure_cfg<SmallCfg>())) return e;
  return configure_cfg<TinyCfg>();
}

namespace {
// k_splitk_reduce over S partial products at P on the C of `d` (S = 0: C = beta C, no partial is read)
cudaError_t launch_reduce(const c128* P, int S, const GemmDesc& d, cudaStream_t stream) {
  const long long tot = (long long)d.M * d.N;
  int blocks = (int)((tot + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  {
    ProfScope scope(stream, "aux.k_splitk_reduce");
    k_splitk_reduce<<<blocks, 256, 0, stream>>>(P, S, d.M, d.N, tot, d);
  }
  count_launch();
  return cudaGetLastError();
}
}  // namespace

cudaError_t zgemm_auto(const GemmDesc& d, const GemmCtx& ctx) {
  if (d.M <= 0 || d.N <= 0 || d.batch <= 0) return cudaSuccess;
  if (d.K <= 0) {
    // BLAS semantics of an empty sum: C = beta C through C's own addressing (beta = 0 writes zeros without reading C);
    // alpha = 0 so that an infinite alpha does not turn the empty sum into NaN
    GemmDesc g = d;
    g.alpha = {0.0, 0.0};
    for (int b = 0; b < d.batch; ++b) {
      g.C = d.C + (long long)b * d.c_batch;
      const cudaError_t e = launch_reduce(nullptr, 0, g, ctx.stream);
      if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
  }
  const GemmPlan pl = plan_gemm(d, ctx);
  GemmDesc g = d;
  g.c_stream = pl.c_stream;
  if (pl.reduce == REDUCE_CLUSTER) {
    g.splitk = pl.S;
    g.k_chunk = pl.k_chunk;
    g.c_split = 0;
    g.cluster_sk = 1;
  } else if (pl.reduce == REDUCE_SCRATCH) {
    g.C = ctx.scratch;
    g.c_m_inner = 1; g.c_m1 = d.N; g.c_m0 = 0; g.c_n = 1; g.c_batch = 0;
    g.alpha = {1.0, 0.0};
    g.beta = {0.0, 0.0};
    g.splitk = pl.S;
    g.k_chunk = pl.k_chunk;
    g.c_split = (long long)d.M * d.N;
  }
  const bool tma = pl.kernel == GEMM_TMA_WIDE || pl.kernel == GEMM_TMA_TALL;
  cudaError_t e = tma ? zgemm_tma_launch(g, pl, ctx) : zgemm_dmma_launch(pl.kernel, g, ctx.stream);
  if (e != cudaSuccess || pl.reduce != REDUCE_SCRATCH) return e;
  return launch_reduce(ctx.scratch, pl.S, d, ctx.stream);
}

}  // namespace tdvp
