// Persistent, TMA-fed variant of the complex128 DMMA GEMM (sm_100a): the big-tile path of zgemm.cu rebuilt around
// cp.async.bulk.tensor + mbarrier, for the GEMMs that carry the D >= 256 work of the sweep
// (H_eff stages 1-3, K_eff, environment updates; reference: opt_einsum -> ZGEMM at pytdscf/_contraction.py:1162-1174).
//
// What changes against zgemm_dmma_kernel<BigCfg> (ncu, profiles/r1_ncu_zgemm_v4_raw.csv: DMMA pipe 90 % busy, the idle
// 10 % being the eight warps leaving the per-k-tile __syncthreads in lock step and queueing on shared memory together):
//  * one producer warp issues TMA boxes into a 4-stage ring; full / empty mbarriers replace every block-wide barrier, so
//    the 8 consumer warps drift apart and their fragment loads interleave with each other's DMMAs;
//  * persistent CTAs (one per SM) walk the tile list, and the producer runs ahead into the next tile while the consumers
//    write the epilogue: prologue / epilogue latency is hidden, no per-tile launch tail;
//  * fragments are double-buffered in registers (loads of step s+1 are issued before the DMMAs of step s);
//  * the complex product runs as a REAL GEMM with doubled k: A' = [re, im] interleaved along k (exactly the memory
//    layout), B're = [re; -im], B'im = [im; re] formed on the fly, so a lane holds ONE double per A row and step
//    (12 fragment doubles per step instead of 20) and conjugation stays a sign-bit flip;
//  * shared memory is written by TMA with the 128-byte hardware swizzle; the k index a lane handles in step t,
//    k = 4 (q >> 1) + t, is chosen so that every LDS phase hits 8 distinct 16-byte bank groups for k-contiguous AND
//    row-contiguous operands (bank arithmetic in DESIGN.md 4.1b).
// Shapes the tensor maps cannot express (batched, rows not a multiple of 8 on a row-contiguous operand, two-level row
// indices that do not tile by 128 / 64) run on the cp.async kernels of zgemm.cu (plan_gemm, zgemm_plan.h).
#include <cuda.h>
#include <cudaTypedefs.h>

#include <mutex>

#include "zgemm_plan.h"

namespace tdvp {

namespace {

constexpr int BK = TMA_BK;
constexpr int CONSUMER_WARPS = 8;
// Registers are allocated per warpgroup (4 warps): 2 consumer warpgroups + 1 producer warpgroup (one working lane).  The
// launch gives every thread 168 registers (65536 / 384); the producer group then shrinks to 40 and the consumers grow
// to 232 with setmaxnreg, as warp-specialised Hopper / Blackwell GEMMs do.
constexpr int THREADS = 32 * (CONSUMER_WARPS + 4);
constexpr int PRODUCER_REGS = 40, CONSUMER_REGS = 232;

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned bar, unsigned parity) {
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
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
__device__ __forceinline__ void tma_load_4d(unsigned dst, const CUtensorMap* map, unsigned bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

__device__ __forceinline__ double flip_sign(double x, unsigned mask) {
  return __hiloint2double(__double2hiint(x) ^ (int)mask, __double2loint(x));
}
__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

template <bool KMAJOR>
__device__ __forceinline__ void issue_box(unsigned dst, const CUtensorMap* map, unsigned bar, const TmaSide& s, int row0, int k0) {
  const int lo = s.small_inner ? 0 : (int)((unsigned)row0 % s.inner);
  const int hi = (int)((unsigned)row0 / s.inner);
  if (KMAJOR) tma_load_4d(dst, map, bar, 2 * k0, s.swapped ? hi : lo, s.swapped ? lo : hi, 0);   // dims (k as f64 pairs, row, outer row, 1)
  else tma_load_4d(dst, map, bar, 0, k0, lo >> 3, hi);                // dims (8 rows as f64 pairs, k, row / 8, outer row)
}

struct Frag {
  double a[4];
  double2 b[4];
};

template <typename C, bool A_KMAJOR, bool B_KMAJOR>
__global__ void __launch_bounds__(THREADS, 1)
    zgemm_tma_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const TmaParams p) {
  constexpr int BM = C::BM, BN = C::BN, STAGES = C::STAGES, SLAB_A = C::SLAB_A, SLAB_B = C::SLAB_B, STAGE_BYTES = C::STAGE_BYTES;
  extern __shared__ unsigned char smem_raw[];
  const unsigned raw = smem_u32(smem_raw);
  const unsigned base = (raw + 1023u) & ~1023u;                  // SWIZZLE_128B pattern repeats every 1024 B of address
  const unsigned char* sm = smem_raw + (base - raw);
  const unsigned bars = base + STAGES * STAGE_BYTES;             // full[STAGES], empty[STAGES]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(bars + 8 * s, 1);
      mbar_init(bars + 8 * (STAGES + s), CONSUMER_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncthreads();
  const int KT_full = (p.K + BK - 1) / BK;
  const int nseg = seg_count(p, KT_full, blockIdx.x, gridDim.x);

  if (warp >= CONSUMER_WARPS) {
    // ================= producer: one lane walks the same work list and keeps the ring full =================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" ::"n"(PRODUCER_REGS));
    if (warp != CONSUMER_WARPS || lane != 0) return;
    asm volatile("prefetch.tensormap [%0];\n" ::"l"(&mapA) : "memory");
    asm volatile("prefetch.tensormap [%0];\n" ::"l"(&mapB) : "memory");
    int stage = 0;
    unsigned phase = 0;
    for (int si = 0; si < nseg; ++si) {
      const Seg sg = get_seg(p, si, KT_full, blockIdx.x, gridDim.x);
      const int tm = sg.tm, tn = sg.tn;
      const int k_begin = sg.split * p.k_chunk;
      for (int kt = sg.kt0; kt < sg.kt1; ++kt) {
        mbar_wait(bars + 8 * (STAGES + stage), phase ^ 1u);      // slot free (passes at once on a fresh barrier)
        const unsigned full = bars + 8 * stage;
        mbar_expect_tx(full, STAGE_BYTES);
        const unsigned sA = base + stage * STAGE_BYTES, sB = sA + 2 * SLAB_A;
        const int k0 = k_begin + kt * BK;
        issue_box<A_KMAJOR>(sA, &mapA, full, p.a, tm * BM, k0);
        issue_box<B_KMAJOR>(sB, &mapB, full, p.b, tn * BN, k0);
        issue_box<A_KMAJOR>(sA + SLAB_A, &mapA, full, p.a, tm * BM, k0 + 8);
        issue_box<B_KMAJOR>(sB + SLAB_B, &mapB, full, p.b, tn * BN, k0 + 8);
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
    return;
  }

  // ================= consumers: 4 x 2 warps of 32 x 32 complex =================
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;\n" ::"n"(CONSUMER_REGS));
  const int g = lane >> 2, q = lane & 3, hq = q >> 1, odd = q & 1;
  const int wm = warp % C::WMW, wn = warp / C::WMW;
  // 16-byte chunk (after the hardware XOR) of the complex k = 4 hq + t this lane handles in step t, for row (or, on
  // row-contiguous operands, 8-row group member) g -- the same value serves both operands and both majors
  int off_t[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) off_t[t] = ((4 * hq + t) ^ g) << 4;
  const int aBase = A_KMAJOR ? ((wm * 32 + g) * 128 + odd * 8) : (wm * 4 * 1024 + 4 * hq * 128 + odd * 8);
  const int bBase = B_KMAJOR ? ((wn * 32 + g) * 128) : (wn * 4 * 1024 + 4 * hq * 128);
  const unsigned maskA = (p.a_conj && odd) ? 0x80000000u : 0u;
  const unsigned maskB = (p.b_conj ? 0x80000000u : 0u) ^ (odd ? 0x80000000u : 0u);

  auto load_frag = [&](Frag& f, const unsigned char* slabA, const unsigned char* slabB, int t) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
      f.a[i] = *reinterpret_cast<const double*>(slabA + aBase + i * 1024 + (A_KMAJOR ? 0 : t * 128) + off_t[t]);
#pragma unroll
    for (int j = 0; j < 4; ++j)
      f.b[j] = *reinterpret_cast<const double2*>(slabB + bBase + j * 1024 + (B_KMAJOR ? 0 : t * 128) + off_t[t]);
  };

  double cre[4][4][2], cim[4][4][2];
  auto compute = [&](const Frag& f) {
    double av[4], bre[4], bim[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) av[i] = flip_sign(f.a[i], maskA);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      // real GEMM over the doubled k: even k' multiplies (b.re | b.im), odd k' multiplies (-b.im | b.re)
      const double y = flip_sign(f.b[j].y, maskB);
      bre[j] = odd ? y : f.b[j].x;
      bim[j] = odd ? f.b[j].x : y;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        dmma(cre[i][j][0], cre[i][j][1], av[i], bre[j]);
        dmma(cim[i][j][0], cim[i][j][1], av[i], bim[j]);
      }
  };

  int stage = 0;
  unsigned phase = 0;
  const c128 alpha = p.alpha, beta = p.beta;
  const bool use_beta = (beta.x != 0.0) || (beta.y != 0.0);
  for (int si = 0; si < nseg; ++si) {
    const Seg sg = get_seg(p, si, KT_full, blockIdx.x, gridDim.x);
    const int tm = sg.tm, tn = sg.tn, split = sg.split;
    const int KT = sg.kt1 - sg.kt0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        cre[i][j][0] = cre[i][j][1] = 0.0;
        cim[i][j][0] = cim[i][j][1] = 0.0;
      }
    Frag f0, f1;
    mbar_wait(bars + 8 * stage, phase);
    load_frag(f0, sm + stage * STAGE_BYTES, sm + stage * STAGE_BYTES + 2 * SLAB_A, 0);
    for (int kt = 0; kt < KT; ++kt) {
      const unsigned char* sA = sm + stage * STAGE_BYTES;
      const unsigned char* sB = sA + 2 * SLAB_A;
      int nstage = stage + 1;
      unsigned nphase = phase;
      if (nstage == STAGES) { nstage = 0; nphase ^= 1u; }
#pragma unroll
      for (int s = 0; s < 8; ++s) {          // s = 4 * slab + t
        Frag& cur = (s & 1) ? f1 : f0;
        Frag& nxt = (s & 1) ? f0 : f1;
        if (s < 7) {
          load_frag(nxt, sA + ((s + 1) >> 2) * SLAB_A, sB + ((s + 1) >> 2) * SLAB_B, (s + 1) & 3);
        } else if (kt + 1 < KT) {
          // first fragments of the next stage are requested before the last DMMAs of this one
          mbar_wait(bars + 8 * nstage, nphase);
          load_frag(nxt, sm + nstage * STAGE_BYTES, sm + nstage * STAGE_BYTES + 2 * SLAB_A, 0);
        }
        compute(cur);
      }
      // every lane's reads of this stage have been consumed by the (warp-synchronous) DMMAs above: hand the slot back
      __syncwarp();
      if (lane == 0) mbar_arrive(bars + 8 * (STAGES + stage));
      stage = nstage;
      phase = nphase;
    }

    if (sg.role >= 2) {
      // ---- stream-K tail / middle part: add the sums the previous CTA published for this tile (fixed order along k) ----
      if (tid == 0) {
        while (*((volatile int*)(p.sk_flags + blockIdx.x - 1)) != p.epoch) {
        }
        __threadfence();
      }
      asm volatile("bar.sync 1, %0;\n" ::"n"(32 * CONSUMER_WARPS) : "memory");
      const c128* ws = p.sk_ws + (size_t)(blockIdx.x - 1) * (BM * BN);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const double2 v = __ldcg(reinterpret_cast<const double2*>(ws + (size_t)((i * 4 + j) * 2 + e) * (32 * CONSUMER_WARPS) + tid));
            cre[i][j][e] = v.x + cre[i][j][e];
            cim[i][j][e] = v.y + cim[i][j][e];
          }
    }
    if (sg.role == 1 || sg.role == 3) {
      // ---- stream-K head / middle part: publish the sums so far (fragment order: 16-byte stores, consecutive lanes) ----
      c128* ws = p.sk_ws + (size_t)blockIdx.x * (BM * BN);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int e = 0; e < 2; ++e)
            ws[(size_t)((i * 4 + j) * 2 + e) * (32 * CONSUMER_WARPS) + tid] = c128{cre[i][j][e], cim[i][j][e]};
      __threadfence();
      asm volatile("bar.sync 1, %0;\n" ::"n"(32 * CONSUMER_WARPS) : "memory");
      if (tid == 0) *((volatile int*)(p.sk_flags + blockIdx.x)) = p.epoch;
      continue;
    }
    // ---- epilogue: C = alpha * acc + beta * C (the producer is already filling the ring for the next tile) ----
    c128* __restrict__ Cg = p.C + (long long)split * p.c_split;
    const int tile_m = tm * BM, tile_n = tn * BN;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = tile_m + wm * 32 + 8 * i + g;
      if (m >= p.M) continue;
      const long long roff = (long long)(m / p.c_m_inner) * p.c_m1 + (long long)(m % p.c_m_inner) * p.c_m0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int n = tile_n + wn * 32 + 8 * j + 2 * q + e;
          if (n >= p.N) continue;
          c128* ptr = Cg + roff + (long long)n * p.c_n;
          const c128 acc = {cre[i][j][e], cim[i][j][e]};
          c128 out = cmul(alpha, acc);
          if (use_beta) out = cadd(out, cmul(beta, *ptr));
          if (p.c_stream) __stcs(reinterpret_cast<double2*>(ptr), make_double2(out.x, out.y));
          else *ptr = out;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host side: tensor maps
// ---------------------------------------------------------------------------------------------------------------
PFN_cuTensorMapEncodeTiled encode_fn() {
  static PFN_cuTensorMapEncodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled>(ptr);
    cudaGetLastError();
  });
  return fn;
}

bool encode(CUtensorMap* map, const c128* ptr, const SidePlan& pl) {
  cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUresult rc = encode_fn()(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 4, const_cast<c128*>(ptr), pl.dims, pl.strides, pl.box, estr,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return rc == CUDA_SUCCESS;
}

template <typename C>
cudaError_t launch_tma(bool ak, bool bk, const CUtensorMap& ma, const CUtensorMap& mb, const TmaParams& p, int grid, cudaStream_t stream) {
  if (ak && bk) zgemm_tma_kernel<C, true, true><<<grid, THREADS, C::SMEM_BYTES, stream>>>(ma, mb, p);
  else if (ak && !bk) zgemm_tma_kernel<C, true, false><<<grid, THREADS, C::SMEM_BYTES, stream>>>(ma, mb, p);
  else if (!ak && bk) zgemm_tma_kernel<C, false, true><<<grid, THREADS, C::SMEM_BYTES, stream>>>(ma, mb, p);
  else zgemm_tma_kernel<C, false, false><<<grid, THREADS, C::SMEM_BYTES, stream>>>(ma, mb, p);
  return cudaGetLastError();
}

template <typename C>
cudaError_t configure_tma() {
  cudaError_t e;
  if ((e = cudaFuncSetAttribute(zgemm_tma_kernel<C, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES))) return e;
  if ((e = cudaFuncSetAttribute(zgemm_tma_kernel<C, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES))) return e;
  if ((e = cudaFuncSetAttribute(zgemm_tma_kernel<C, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES))) return e;
  return cudaFuncSetAttribute(zgemm_tma_kernel<C, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
}

}  // namespace

cudaError_t zgemm_tma_configure_device(GemmCtx& ctx) {
  ctx.tma_encode = encode_fn() != nullptr;
  cudaError_t e;
  if ((e = configure_tma<WideCfg>())) return e;
  return configure_tma<TallCfg>();
}

cudaError_t zgemm_tma_launch(const GemmDesc& d, const GemmPlan& pl, const GemmCtx& ctx) {
  CUtensorMap ma, mb;
  if (!encode(&ma, d.A, pl.a_map) || !encode(&mb, d.B, pl.b_map)) return zgemm_dmma_launch(GEMM_BIG, d, ctx.stream);
  TmaParams p;
  p.M = d.M; p.N = d.N; p.K = d.K;
  p.tiles_m = pl.tiles_m; p.tiles_n = pl.tiles_n; p.group_m = pl.group_m;
  p.splitk = d.splitk; p.k_chunk = d.k_chunk;
  p.a = pl.a; p.b = pl.b;
  p.a_conj = d.a_conj ? 1u : 0u;
  p.b_conj = d.b_conj ? 1u : 0u;
  p.C = d.C; p.c_m_inner = d.c_m_inner; p.c_m1 = d.c_m1; p.c_m0 = d.c_m0; p.c_n = d.c_n; p.c_split = d.c_split;
  p.alpha = d.alpha; p.beta = d.beta; p.c_stream = d.c_stream;
  p.streamk = pl.streamk; p.sk_tiles = pl.sk_tiles;
  p.sk_flags = ctx.sk_flags;
  p.sk_ws = ctx.sk_ws;
  p.epoch = p.streamk ? ++ctx.sk_epoch : 0;
  cudaError_t e;
  {
    ProfScope scope(ctx.stream, d.tag, 8.0 * (double)d.M * (double)d.N * (double)d.K, true);
    e = pl.kernel == GEMM_TMA_TALL ? launch_tma<TallCfg>(pl.a_kmajor, pl.b_kmajor, ma, mb, p, pl.grid, ctx.stream)
                                   : launch_tma<WideCfg>(pl.a_kmajor, pl.b_kmajor, ma, mb, p, pl.grid, ctx.stream);
  }
  count_launch();
  return e;
}

}  // namespace tdvp
