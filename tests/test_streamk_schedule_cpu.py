"""The ZGEMM launch planner (pytdscf_b200/csrc/zgemm_plan.h) on the CPU, called through tests/c/gemm_plan_shim.cpp built with g++.

The stream-K work assignment (``seg_count`` / ``get_seg``, the functions zgemm_tma_kernel runs) and the rule that sets
``streamk`` / ``sk_tiles`` / the grid are checked for the properties the kernel relies on: every (tile, k-tile) is computed
exactly once; a tile cut over several CTAs is published by CTA c and continued by CTA c + 1 (never a CTA with a lower index
waiting for a higher one: in-order CTA dispatch then makes the wait deadlock-free); a CTA publishes at most once per launch
(one partial buffer and one flag per CTA) and does so BEFORE anything it waits for.  ``plan_gemm`` is checked over a shape
grid for the conditions each kernel and reduction needs.  The GPU tests (tests/test_gpu_bench_shapes.py) pin the kernels."""
import ctypes
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
G_SMS = 148
SCRATCH_ELEMS = 18 << 20                     # SPLITK_SCRATCH_ELEMS
GEMM_BIG, GEMM_SMALL, GEMM_TINY, GEMM_TMA_WIDE, GEMM_TMA_TALL = 1, 2, 3, 4, 5
REDUCE_NONE, REDUCE_CLUSTER, REDUCE_SCRATCH = 0, 1, 2
TILE = {GEMM_BIG: (128, 64, 16), GEMM_SMALL: (64, 32, 8), GEMM_TINY: (32, 32, 8), GEMM_TMA_WIDE: (128, 64, 16),
        GEMM_TMA_TALL: (256, 32, 16)}          # BM, BN, BK
PLAN_FIELDS = ("kernel", "S", "k_chunk", "reduce", "c_stream", "tiles_m", "tiles_n", "group_m", "streamk", "sk_tiles", "grid")

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")

LL = ctypes.c_longlong
P_LL = ctypes.POINTER(LL)
P_INT = ctypes.POINTER(ctypes.c_int)


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("gemm_plan") / "gemm_plan_shim.so")
    cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-Werror", "-fPIC", "-shared", "-I", os.path.join(ROOT, "pytdscf_b200", "csrc"),
           "-I", os.path.join(CUDA, "include"), os.path.join(ROOT, "tests", "c", "gemm_plan_shim.cpp"), "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    lib = ctypes.CDLL(so)
    lib.gemm_plan.argtypes = [P_LL, P_LL, P_LL]
    lib.gemm_plan_streamk.argtypes = [LL, ctypes.c_int, P_LL, P_LL]
    lib.gemm_plan_side_ok.argtypes = [LL, LL, ctypes.c_int, ctypes.c_int, LL, LL, LL, ctypes.c_int]
    lib.gemm_plan_segments.argtypes = [ctypes.c_int] * 10 + [P_INT, ctypes.c_int]
    return lib


def ctx_arr(force_cfg=0, force_splitk=0, force_cstream=0):
    """Context of a B200 handle: split-K scratch, stream-K buffers for every SM, tensor-map encoder found."""
    return (LL * 9)(1, SCRATCH_ELEMS, G_SMS, force_cfg, force_splitk, force_cstream, 1, G_SMS, 1)


def plan(shim, desc, **ctx):
    out = (LL * 11)()
    shim.gemm_plan((LL * 14)(*desc), ctx_arr(**ctx), out)
    return dict(zip(PLAN_FIELDS, out))


def host_rule(shim, total: int, KT: int, force_tma: bool = False):
    """-> (streamk, sk_tiles, grid) of `total` single-split tiles of KT k-tiles; force_tma: tdvp_set_gemm_config tile 4."""
    out = (LL * 3)()
    shim.gemm_plan_streamk(total, KT, ctx_arr(force_cfg=4 if force_tma else 0), out)
    return tuple(out)


def kernel_segments(shim, cta, grid, tiles_m, tiles_n, splitk, K, k_chunk, group_m, streamk, sk_tiles):
    """-> [(tm, tn, split, kt0, kt1, role)] in execution order: get_seg for si = 0 .. seg_count - 1."""
    cap = tiles_m * tiles_n * splitk + 2
    buf = (ctypes.c_int * (6 * cap))()
    n = shim.gemm_plan_segments(tiles_m, tiles_n, splitk, K, k_chunk, group_m, streamk, sk_tiles, cta, grid, buf, cap)
    assert 0 <= n <= cap
    return [tuple(buf[6 * i:6 * i + 6]) for i in range(n)]


def segments(shim, cta: int, grid: int, total: int, KT: int, streamk: int, sk_tiles: int):
    """-> [(tile, kt0, kt1, role)]: with a single column of tiles the raster order is the tile index itself."""
    out = []
    for tm, tn, split, k0, k1, role in kernel_segments(shim, cta, grid, total, 1, 1, 16 * KT, 0, 8, streamk, sk_tiles):
        assert tn == 0 and split == 0
        out.append((tm, k0, k1, role))
    return out


CASES = [(t, kt, f) for f in (False, True) for kt in (16, 17, 32, 64, 96, 512) for t in
         (1, 8, 40, 73, 74, 80, 96, 147, 148, 149, 150, 216, 295, 296, 297, 384, 512, 1024, 4096, 4097)]


@pytest.mark.parametrize("total,KT,force", CASES)
def test_streamk_assignment_properties(shim, total, KT, force):
    streamk, sk_tiles, grid = host_rule(shim, total, KT, force_tma=force)
    assert 1 <= grid <= G_SMS
    covered = {}
    publisher, continuer = {}, {}
    for cta in range(grid):
        segs = segments(shim, cta, grid, total, KT, streamk, sk_tiles)
        publishes = [s for s in segs if s[3] in (1, 3)]
        assert len(publishes) <= 1                                  # one partial buffer / flag per CTA and launch
        waited = False
        for tile, k0, k1, role in segs:
            assert 0 <= tile < total and 0 <= k0 < k1 <= KT
            for k in range(k0, k1):
                assert (tile, k) not in covered, (tile, k)
                covered[(tile, k)] = cta
            if role in (2, 3):
                waited = True
                continuer.setdefault(tile, []).append((cta, k0, k1))
            if role == 1:
                assert not waited                                    # a head is published before this CTA waits for anything
            if role in (1, 3):
                publisher.setdefault(tile, []).append((cta, k0, k1))
            if role == 1:
                assert k0 == 0
            if role == 2:
                assert k1 == KT
    assert len(covered) == total * KT                                # everything exactly once
    for tile, cont in continuer.items():
        for cta, k0, _ in cont:                                      # the CTA that continues a tile reads its predecessor's buffer
            prev = [p for p in publisher.get(tile, []) if p[2] == k0]
            assert prev and prev[0][0] == cta - 1, (tile, cta, prev)
    for tile, pubs in publisher.items():
        for cta, _, k1 in pubs:                                      # every published partial is picked up
            assert any(c[1] == k1 and c[0] == cta + 1 for c in continuer.get(tile, [])), (tile, cta)
    if not force:
        chain = max((len(v) for v in publisher.values()), default=0)
        assert chain <= 2                                            # zgemm_auto: at most two hand-overs (three CTAs) per tile
        if total >= G_SMS:
            assert chain <= 1                                        # ranges of at least one tile: two CTAs per tile
        if streamk and total >= 2 * G_SMS:
            assert G_SMS < sk_tiles < 2 * G_SMS                      # one to two waves' worth, the rest in whole waves


A_ADDR, B_ADDR = 1 << 32, 3 << 31


def operands(layout, M, N, K, inner):
    """(a_m_inner, a_m1, a_m0, a_k, b_n_inner, b_n1, b_n0, b_k) of a row-major GEMM (NN / NT / TN / CN) or of a two-level A
    as contract.cu builds it (2k: k-contiguous rows m = (c, w) of an environment, 2r: row-contiguous H_eff stage 2)."""
    b = (1, K, 0, 1) if layout == "NT" else (1, 1, 0, N)
    if layout in ("NN", "NT"):
        return (1, K, 0, 1) + b
    if layout in ("TN", "CN"):
        return (1, 1, 0, M) + b
    if layout == "2k":
        return (inner, inner, 4 * inner, 1) + b
    return (inner, 12 * inner, 1, inner) + b


SHAPES = [(M, N, K, layout, inner, batch)
          for M in (1, 8, 33, 64, 100, 256, 500, 1024, 1536, 4096, 8192, 37888)
          for N in (1, 8, 32, 33, 100, 256, 1024, 4096, 8192)
          for K in (1, 16, 17, 64, 256, 512, 1000, 4096)
          for layout, inner in (("NN", 1), ("NT", 1), ("TN", 1), ("CN", 1), ("2k", 64), ("2k", 100), ("2r", 64), ("2r", 10))
          for batch in (1, 3)]


def test_plan_invariants_automatic_mode(shim):
    n_tma = n_cluster = n_scratch = n_streamk = 0
    for M, N, K, layout, inner, batch in SHAPES:
        a_in, a1, a0, ak, b_in, b1, b0, bk = operands(layout, M, N, K, inner)
        desc = (M, N, K, batch, A_ADDR, a_in, a1, a0, ak, B_ADDR, b_in, b1, b0, bk)
        p = plan(shim, desc)
        kern, S, chunk, red = p["kernel"], p["S"], p["k_chunk"], p["reduce"]
        case = (M, N, K, layout, inner, batch, p)
        BM, BN, BK = TILE[kern]
        if kern in (GEMM_TMA_WIDE, GEMM_TMA_TALL):                   # tensor maps describe both operands
            n_tma += 1
            assert batch == 1, case
            assert shim.gemm_plan_side_ok(A_ADDR, M, K, a_in, a1, a0, ak, BM), case
            assert shim.gemm_plan_side_ok(B_ADDR, N, K, b_in, b1, b0, bk, BN), case
            assert (p["tiles_m"], p["tiles_n"]) == (-(-M // BM), -(-N // BN)), case
            assert 8 <= p["group_m"] <= 64, case
        assert (red == REDUCE_NONE) == (S == 1), case
        if red == REDUCE_CLUSTER:                                    # a cluster of S small / tiny CTAs per tile
            n_cluster += 1
            assert kern in (GEMM_SMALL, GEMM_TINY) and 2 <= S <= 16 and batch == 1, case
        if red == REDUCE_SCRATCH:                                    # the partials fit the split-K scratch
            n_scratch += 1
            assert S * M * N <= SCRATCH_ELEMS, case
        assert chunk % BK == 0 and (S - 1) * chunk < K <= S * chunk, case   # S chunks of whole k-tiles cover K exactly
        if p["streamk"]:
            n_streamk += 1
            assert kern in (GEMM_TMA_WIDE, GEMM_TMA_TALL) and S == 1 and -(-K // 16) >= 16, case
            assert p["grid"] <= G_SMS, case
        if S == 1:
            assert p["c_stream"] == (M * N * batch * 16 > 64e6), case   # evict-first stores for outputs above half of L2
        else:
            assert p["c_stream"] == 0, case
    assert min(n_tma, n_cluster, n_scratch, n_streamk) > 0           # the grid reaches every kind of plan


@pytest.mark.parametrize("M,N,K,layout", [(1280, 2560, 256, "NN"), (8192, 4096, 1024, "NN"), (1024, 1024, 4096, "TN"),
                                          (40000, 32, 512, "NN"), (37888, 16, 256, "2r"), (512, 512, 8192, "CN")])
@pytest.mark.parametrize("force_cfg,force_splitk", [(0, 0), (0, 1), (4, 0), (4, 1), (5, 1), (0, 3)])
def test_planned_schedule_covers_the_work_once(shim, M, N, K, layout, force_cfg, force_splitk):
    """The TMA plans of real shapes (2-D rasters, grouped order, split-K items) are executed exactly once by the kernel's
    work assignment."""
    inner = 64 if layout == "2r" else 1
    a_in, a1, a0, ak, b_in, b1, b0, bk = operands(layout, M, N, K, inner)
    p = plan(shim, (M, N, K, 1, A_ADDR, a_in, a1, a0, ak, B_ADDR, b_in, b1, b0, bk), force_cfg=force_cfg, force_splitk=force_splitk)
    if p["kernel"] not in (GEMM_TMA_WIDE, GEMM_TMA_TALL):
        assert force_cfg == 0                                        # forced tma always gets the TMA kernel for these shapes
        return
    S, chunk, KT = p["S"], p["k_chunk"], -(-K // 16)
    seen, count = set(), 0
    for cta in range(p["grid"]):
        for tm, tn, split, k0, k1, _ in kernel_segments(shim, cta, p["grid"], p["tiles_m"], p["tiles_n"], S, K, chunk,
                                                        p["group_m"], p["streamk"], p["sk_tiles"]):
            assert 0 <= tm < p["tiles_m"] and 0 <= tn < p["tiles_n"] and 0 <= split < S
            seen.update((tm, tn, split, k) for k in range(k0, k1))
            count += k1 - k0
    per_split = [-(-min(chunk, K - s * chunk) // 16) for s in range(S)] if S > 1 else [KT]
    assert count == len(seen) == p["tiles_m"] * p["tiles_n"] * sum(per_split)   # every (tile, split, k-tile) exactly once
