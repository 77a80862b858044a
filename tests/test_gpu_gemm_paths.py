"""Every ZGEMM kernel on the operand layouts its planner accepts, driven through the library's own ``tdvp::gemm`` with
arbitrary ``GemmDesc`` descriptors (tests/c/gemm_desc_shim.cpp, linked against the loaded libtdvp_b200.so).

Each case
- embeds A, B and C in larger buffers filled with one NaN bit pattern: A and B must come back bitwise unchanged, every C
  element the descriptor does not address must still hold the pattern, and with beta = 0 the addressed C elements start
  as that NaN (a kernel that reads C then fails);
- in exact mode uses integer re / im parts in [-4, 4] and dyadic alpha / beta, so every partial sum is exact in fp64 in
  any order and the result must equal the NumPy float64 reference bit for bit;
- in graded mode scales the rows of A and the columns of B over 2^-40 .. 2^40 and bounds each element's error against a
  long-double reference by 4 (K + 2) 2^-53 (|alpha| |A| |B| + |beta| |C0|);
- asserts the plan (kernel, split-K factor, reduction, stream-K, tensor-map geometry) and checks with torch.profiler
  that the kernel instantiation that ran is the planned one, with k_splitk_reduce exactly when the reduction is scratch.

The production descriptor builders are replicated from the same formulas: left_apply_skip (contract.cu:152-157),
stage2_full (contract.cu:196-199), heff2_mid's row chunks (contract.cu:381-387), vhc_desc (qr.cu:557-564) and the pinv
GEMM (svd.cu:749-750)."""
import collections
import ctypes
import os
import re
import shutil
import subprocess
from dataclasses import dataclass, field

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu      # every test here but the case-table check needs the device

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
POISON = np.uint64(0x7FF8DEADBEEFCAFE)        # a quiet NaN with a payload no computation produces
FRONT, BACK = 8, 64                           # poisoned guard elements before / after each operand
BIG, SMALL, TINY, WIDE, TALL = 1, 2, 3, 4, 5
NONE, CLUSTER, SCRATCH = 0, 1, 2
KNAME = {BIG: "big", SMALL: "small", TINY: "tiny", WIDE: "tma-wide", TALL: "tma-tall"}
RNAME = {NONE: "none", CLUSTER: "cluster", SCRATCH: "scratch"}
CFG_ARGS = {BIG: "4, 2, 16, 3, 4, 4", SMALL: "2, 1, 8, 4, 4, 4", TINY: "2, 2, 8, 3, 2, 2", WIDE: "4, 2, 4", TALL: "8, 1, 3"}
PLAN_FIELDS = ("kernel", "S", "k_chunk", "reduce", "c_stream", "tiles_m", "tiles_n", "group_m", "streamk", "sk_tiles", "grid",
               "a_kmajor", "b_kmajor", "a_small", "a_swapped", "b_small", "b_swapped")
TILE_CFG = {"auto": 0, "big": 1, "small": 2, "tiny": 3, "tma": 4, "tma_tiles": 5}
EXACT_ALPHA, EXACT_BETA = 2 - 1j, 0.5 + 1.5j
GRADED_ALPHA, GRADED_BETA = 0.7 - 0.2j, -0.3 + 0.5j


# ---- fixtures ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng():
    from pytdscf_b200._engine import Engine

    e = Engine(0)
    yield e
    e.set_gemm_config("auto", 0, 0)
    e.close()


@pytest.fixture(scope="module")
def shim(eng, tmp_path_factory):
    """tests/c/gemm_desc_shim.cpp built with g++ against the library instance the Engine loaded (linked by path, with an
    rpath to its directory, so the loader binds the shim to that same instance)."""
    from pytdscf_b200 import _lib

    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    lib_path = _lib.LIB_PATH
    so = str(tmp_path_factory.mktemp("gemm_desc") / "gemm_desc_shim.so")
    cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-Werror", "-fPIC", "-shared", "-I", os.path.join(ROOT, "pytdscf_b200", "csrc"),
           "-I", os.path.join(CUDA, "include"), os.path.join(ROOT, "tests", "c", "gemm_desc_shim.cpp"), lib_path,
           "-Wl,-rpath," + os.path.dirname(lib_path), "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    lib = ctypes.CDLL(so)
    lib.gemm_desc_run.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_longlong), ctypes.POINTER(ctypes.c_double),
                                  ctypes.POINTER(ctypes.c_longlong)]
    lib.gemm_desc_run.restype = ctypes.c_int
    # the same library instance: a launch through the shim shows in the Engine's launch counter
    a, c = (torch.zeros(64, dtype=torch.complex128, device="cuda") for _ in range(2))
    before = eng.stats()["launches"]
    desc = (8, 8, 8, a.data_ptr(), 1, 8, 0, 1, 0, a.data_ptr(), 1, 1, 0, 8, 0, c.data_ptr(), 1, 8, 0, 1)
    out = (ctypes.c_longlong * len(PLAN_FIELDS))()
    assert lib.gemm_desc_run(eng.h, (ctypes.c_longlong * 20)(*desc), (ctypes.c_double * 4)(1, 0, 0, 0), out) == 0
    torch.cuda.synchronize()
    assert eng.stats()["launches"] > before
    return lib


# ---- operand layouts -----------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Op:
    """One operand of `rows` rows (two-level: row = r1 * inner + r0) and `cols` columns, element (row, col) at
    r1 * s1 + r0 * s0 + col * sc."""
    inner: int
    s1: int
    s0: int
    sc: int
    label: str


def operand(kind, rows, K, inner=1, R=128):
    """A / B operand layouts.  k: k-contiguous rows (lda > K); row: row-contiguous (the k stride > rows); k2 / k2d:
    two-level k-contiguous with ascending (s0 < s1) / descending (s0 > s1, left_apply_skip's form) strides; r2: two-level
    row-contiguous (stage2_full's form).  The label names the tensor-map geometry for tile rows R."""
    if kind == "k":
        return Op(1, K + 3, 0, 1, "k-major")
    if kind == "row":
        return Op(1, 1, 0, rows + 5, "row" if rows % 8 == 0 else "row-ragged")
    n1 = rows // inner
    assert n1 * inner == rows and n1 > 1
    tile = inner % R == 0 or R % inner == 0
    if kind == "k2":
        s0 = K + 2
        label = f"k2-{inner // R}R" if inner % R == 0 else (f"k2-small{inner}" if tile else f"untileable{inner}")
        return Op(inner, inner * s0 + 7, s0, 1, label)
    if kind == "k2d":
        s1 = K + 1
        label = ("swapped" if inner >= R else f"k2-small{inner}-desc") if tile else f"untileable{inner}"
        return Op(inner, s1, n1 * s1 + 3, 1, label)
    if kind == "r2":
        return Op(inner, K * inner + 8, 1, inner, "r2" if inner >= R else "r2-small")
    raise ValueError(kind)


def c_layout(kind, M, N, inner=1):
    """C layouts: row (ldc > N), s2 (stage2_full: rows (a, s), s contiguous, n stride Dr), las (left_apply_skip: rows
    (channel, a), a stride w * ncols), col (vhc_desc: column-major)."""
    if kind == "row":
        return Op(1, N + 3, 0, 1, "row")
    if kind == "s2":
        return Op(inner, N * inner + 5, 1, inner, "stage2_full")
    if kind == "las":
        return Op(inner, N + 2, (M // inner) * (N + 2) + 1, 1, "left_apply_skip")
    if kind == "col":
        return Op(1, 1, 0, M + 4, "column-major")
    raise ValueError(kind)


def custom(inner, s1, s0, sc, label):
    return Op(inner, s1, s0, sc, label)


@dataclass
class Case:
    name: str
    M: int
    N: int
    K: int
    a: Op
    b: Op
    c: Op
    cfg: tuple                       # tdvp_set_gemm_config (tile, splitk, c_stream)
    kernel: int
    reduce: int
    S: int = 1
    streamk: int | None = None       # expected plan streamk (None: not checked)
    conj: tuple = (0, 0)
    beta0: bool = False
    mode: str = "exact"
    chunks: tuple = ()               # heff2_mid: row chunks (in units of a_m_inner rows) run as separate calls
    flags: dict = field(default_factory=dict)

    @property
    def id(self):
        cj = "".join("c" if x else "-" for x in self.conj)
        return (f"{self.name}:{KNAME[self.kernel]}-{RNAME[self.reduce]}{self.S if self.S > 1 else ''}"
                f"-A[{self.a.label}]-B[{self.b.label}]-C[{self.c.label}]-{self.M}x{self.N}x{self.K}"
                f"-{self.cfg[0]}.S{self.cfg[1]}.cs{self.cfg[2]}-conj{cj}-{'b0' if self.beta0 else 'b1'}-{self.mode}")


def mk(name, M, N, K, a, b, c, cfg, kernel, reduce, S=1, **kw):
    R_A, R_B = (256, 32) if kernel == TALL else (128, 64)
    A = a if isinstance(a, Op) else operand(a[0], M, K, *a[1:2], R=R_A)
    B = b if isinstance(b, Op) else operand(b[0], N, K, *b[1:2], R=R_B)
    C = c if isinstance(c, Op) else c_layout(c[0], M, N, *c[1:2])
    return Case(name, M, N, K, A, B, C, cfg, kernel, reduce, S, **kw)


T = ("tma", 1, 0)
CASES = [
    # cp.async kernels: tails at BM / BN +- 1, K in {1, 15, 16, 17}, forced c_stream, conjugation
    mk("big-tail+", 129, 65, 17, ("k",), ("row",), ("row",), ("big", 1, 2), BIG, NONE),
    mk("big-tail-", 127, 63, 15, ("row",), ("k",), ("col",), ("big", 1, 1), BIG, NONE, conj=(1, 0), beta0=True, mode="graded"),
    mk("big-untileable", 192, 200, 40, ("k2", 96), ("k2", 100), ("s2", 64), ("tma", 1, 0), BIG, NONE),
    mk("big-untileable-desc", 200, 192, 33, ("k2d", 100), ("k2d", 96), ("las", 40), ("tma", 1, 2), BIG, NONE, beta0=True),
    mk("small-tail+", 65, 31, 1, ("row",), ("row",), ("row",), ("small", 1, 2), SMALL, NONE, conj=(0, 1), beta0=True),
    mk("small-tail-", 63, 33, 15, ("k",), ("k",), ("col",), ("small", 1, 1), SMALL, NONE, conj=(0, 1), mode="graded"),
    mk("tiny-tail", 31, 33, 17, ("row",), ("k",), ("row",), ("tiny", 1, 2), TINY, NONE, beta0=True),
    mk("tiny-tail2", 33, 31, 16, ("k",), ("row",), ("col",), ("tiny", 1, 1), TINY, NONE, conj=(1, 1), mode="graded"),
    mk("tiny-K1", 33, 33, 1, ("k",), ("k",), ("row",), ("tiny", 1, 0), TINY, NONE, conj=(1, 0)),
    # split-K through a thread-block cluster
    mk("small-cluster2", 128, 64, 200, ("k2d", 32), ("k2", 32), ("las", 32), ("small", 2, 0), SMALL, CLUSTER, 2),
    mk("tiny-cluster2", 96, 64, 65, ("r2", 32), ("row",), ("s2", 32), ("tiny", 2, 2), TINY, CLUSTER, 2, conj=(1, 0),
       beta0=True, mode="graded"),
    mk("tiny-cluster16", 64, 32, 639, ("k",), ("k2", 8), ("row",), ("tiny", 16, 0), TINY, CLUSTER, 16, beta0=True),
    mk("small-cluster16", 64, 33, 1024, ("row",), ("k",), ("col",), ("small", 16, 2), SMALL, CLUSTER, 16, conj=(0, 1),
       mode="graded"),
    # split-K through the scratch buffer and k_splitk_reduce
    mk("big-scratch4", 256, 64, 513, ("k2d", 128), ("row",), ("las", 64), ("big", 4, 0), BIG, SCRATCH, 4),
    mk("big-scratch4-tail", 127, 65, 575, ("row",), ("k",), ("col",), ("big", 4, 1), BIG, SCRATCH, 4, conj=(0, 1),
       beta0=True, mode="graded"),
    mk("tma-scratch2", 256, 256, 257, ("k2", 128), ("k2", 128), ("s2", 128), ("tma", 2, 0), WIDE, SCRATCH, 2, beta0=True),
    mk("tma-scratch2-tail", 129, 65, 256, ("k",), ("k",), ("row",), ("tma", 2, 1), WIDE, SCRATCH, 2, conj=(1, 0),
       mode="graded"),
    mk("tiny-scratch3", 32, 32, 97, ("k2", 8), ("row",), ("s2", 8), ("tiny", 3, 1), TINY, SCRATCH, 3, beta0=True),
    mk("tiny-scratch3-tail", 33, 31, 119, ("k",), ("k",), ("col",), ("tiny", 3, 1), TINY, SCRATCH, 3, conj=(1, 1),
       mode="graded"),
    # TMA wide: stream-K in automatic mode (ragged shapes), forced 4 (long chains), forced 5 (whole tiles only)
    mk("sk-auto", 1280, 960, 512, ("k",), ("row",), ("row",), ("auto", 0, 0), WIDE, NONE, streamk=1),
    mk("sk-auto-ragged", 2500, 1100, 1000, ("k",), ("k",), ("col",), ("auto", 0, 2), WIDE, NONE, streamk=1, beta0=True),
    mk("sk-chain", 256, 128, 1024, ("r2", 64), ("row",), ("s2", 64), ("tma", 1, 0), WIDE, NONE, streamk=1, beta0=True),
    mk("sk-chain-tail", 200, 72, 273, ("k",), ("k",), ("row",), ("tma", 1, 1), WIDE, NONE, streamk=1, conj=(1, 0),
       mode="graded"),
    mk("tiles-only", 512, 192, 64, ("k2", 256), ("k2d", 64), ("las", 128), ("tma_tiles", 1, 0), WIDE, NONE, streamk=0),
    mk("tiles-only-tail", 127, 65, 16, ("k",), ("k",), ("col",), ("tma_tiles", 1, 2), WIDE, NONE, streamk=0, conj=(0, 1),
       beta0=True, mode="graded"),
    # TMA wide: every tensor-map geometry of A and B
    mk("wide-small64", 512, 128, 48, ("k2", 64), ("r2", 64), ("row",), ("tma", 1, 2), WIDE, NONE, streamk=0, beta0=True),
    mk("wide-las64", 256, 64, 32, ("k2d", 64), ("r2", 32), ("las", 64), T, WIDE, NONE, streamk=0),
    mk("wide-small8-desc", 256, 64, 17, ("k2d", 8), ("row",), ("row",), ("tma", 1, 1), WIDE, NONE, streamk=0, beta0=True,
       mode="graded"),
    mk("wide-small32", 256, 128, 16, ("k2", 32), ("k2d", 32), ("s2", 32), T, WIDE, NONE, streamk=0, conj=(1, 1)),
    mk("wide-r2", 512, 128, 20, ("r2", 256), ("k2", 64), ("col",), ("tma", 1, 2), WIDE, NONE, streamk=0, mode="graded"),
    mk("wide-swapped2R", 512, 96, 33, ("k2d", 256), ("k2", 32), ("row",), T, WIDE, NONE, streamk=0, beta0=True),
    mk("wide-swapped1R", 256, 64, 24, ("k2d", 128), ("k2d", 8), ("las", 128), ("tma_tiles", 1, 0), WIDE, NONE, streamk=0,
       conj=(0, 1)),
    mk("wide-r2-small16", 256, 256, 40, ("r2", 16), ("k2d", 128), ("s2", 16), T, WIDE, NONE, streamk=0, beta0=True,
       mode="graded"),
    mk("wide-small8", 128, 128, 16, ("k2", 8), ("k2", 64), ("row",), T, WIDE, NONE, streamk=0, conj=(1, 0)),
    mk("wide-small32-desc", 256, 64, 64, ("k2d", 32), ("k2", 8), ("col",), T, WIDE, NONE, streamk=0, conj=(0, 1),
       mode="graded"),
    mk("wide-row", 256, 128, 32, ("row",), ("k2d", 32), ("row",), T, WIDE, NONE, streamk=0, conj=(1, 1), beta0=True),
    mk("wide-small8-desc-2R", 256, 256, 32, ("k2d", 8), ("k2", 128), ("row",), T, WIDE, NONE, streamk=0, conj=(0, 1)),
    mk("wide-small64-r2small", 256, 128, 16, ("k2", 64), ("r2", 32), ("s2", 64), ("tma", 1, 2), WIDE, NONE, streamk=0,
       beta0=True, mode="graded"),
    mk("wide-1R-r2", 256, 256, 24, ("k2", 128), ("r2", 128), ("las", 128), T, WIDE, NONE, streamk=0),
    mk("wide-small32-b-desc8", 256, 64, 40, ("k2", 32), ("k2d", 8), ("col",), T, WIDE, NONE, streamk=0, beta0=True,
       mode="graded"),
    mk("big-untileable-2", 192, 200, 24, ("k2d", 96), ("k2", 100), ("col",), ("tma_tiles", 1, 0), BIG, NONE, conj=(1, 0)),
    mk("small-untileable", 300, 192, 24, ("k2", 100), ("k2d", 96), ("row",), ("small", 1, 0), SMALL, NONE, beta0=True,
       mode="graded"),
    # TMA tall (N <= 32 and M >= 256 * 148): its B has 32-row tiles, so two-level B rows are always smaller than a tile
    mk("tall-tail", 37889, 31, 16, ("k",), ("k",), ("row",), ("tma", 1, 2), TALL, NONE, streamk=0),
    mk("tall-r2-small", 38400, 32, 17, ("r2", 64), ("row",), ("s2", 64), ("tma_tiles", 1, 0), TALL, NONE, streamk=0,
       beta0=True),
    mk("tall-small-desc", 38400, 32, 48, ("k2d", 32), ("k2", 16), ("las", 32), ("tma", 1, 1), TALL, NONE, streamk=0,
       conj=(1, 0)),
    mk("tall-swapped", 38400, 32, 16, ("k2d", 256), ("k2d", 8), ("row",), T, TALL, NONE, streamk=0),
    mk("tall-k2-2R", 38400, 32, 24, ("k2", 512), ("r2", 16), ("col",), T, TALL, NONE, streamk=0, beta0=True, conj=(0, 1)),
    mk("tall-small8", 38400, 32, 16, ("k",), ("k2", 8), ("row",), T, TALL, NONE, streamk=0),
    mk("tall-small64-desc", 38400, 32, 20, ("k2d", 64), ("k2", 8), ("s2", 64), ("tma", 1, 2), TALL, NONE, streamk=0,
       beta0=True),
    mk("tall-b-desc8", 38400, 24, 32, ("k",), ("k2d", 8), ("las", 64), T, TALL, NONE, streamk=0, conj=(0, 1)),
    mk("tall-row", 37888, 16, 16, ("row",), ("k",), ("col",), T, TALL, NONE, streamk=0, conj=(0, 1)),
    mk("tall-1R-small16", 38400, 32, 16, ("k2", 256), ("k2", 16), ("row",), T, TALL, NONE, streamk=0, beta0=True),
    mk("tall-r2", 38912, 24, 32, ("r2", 1024), ("r2", 8), ("row",), ("tma", 1, 2), TALL, NONE, streamk=0, conj=(1, 1)),
]


# ---- replicas of the production descriptor builders ------------------------------------------------------------------
def left_apply_skip_case(D, w, c0, c1, ncols, cfg, kernel, reduce, S=1, **kw):
    """contract.cu:152-157: A = L[:, c0:c1, :] with rows (channel, a), B = X (row-contiguous, ld ncols), C rows (channel, a)
    of a (D, w, ncols) tensor.  The buffers hold the whole L / C, so the skipped channels stay poisoned."""
    M = D * (c1 - c0)
    lbl = "k2-small%d-desc" % D if D < 128 else "swapped"
    A = custom(D, D, w * D, 1, lbl)
    B = custom(1, 1, 0, ncols, "row")
    C = custom(D, ncols, w * ncols, 1, "left_apply_skip")
    return Case(f"left_apply_skip-D{D}", M, ncols, D, A, B, C, cfg, kernel, reduce, S, flags={"a_off": c0 * D, "c_off": c0 * ncols},
                **kw)


def stage2_full_case(Dl, wl, d, wr, Dr, cfg, kernel, reduce, S=1, chunks=(), **kw):
    """contract.cu:196-199: T2[a,i,t,s] = sum_cj Wp[(c,j),(i,t)] T1[a,c,j,s]: A rows (a, s) with s contiguous and k stride
    Dr, B = Wp row-contiguous (ld d wr), C rows (a, s) with n stride Dr."""
    R = 256 if kernel == TALL else 128
    A = custom(Dr, wl * d * Dr, 1, Dr, "r2" if Dr >= R else "r2-small")
    B = custom(1, 1, 0, d * wr, "row" if (d * wr) % 8 == 0 else "row-ragged")
    C = custom(Dr, d * wr * Dr, 1, Dr, "stage2_full")
    name = f"heff2_mid-chunks{len(chunks)}-Dr{Dr}" if chunks else f"stage2_full-Dr{Dr}"
    return Case(name, Dl * Dr, d * wr, wl * d, A, B, C, cfg, kernel, reduce, S, chunks=chunks, **kw)


def vhc_case(jb, nc, mp, ld, cfg, kernel, reduce, S=1, **kw):
    """qr.cu:557-564: W^T = C^T conj(V): A = C panel (row-contiguous, k stride ld), B = V (row-contiguous, conj), C = W
    column-major with ld nc."""
    A = custom(1, 1, 0, ld, "row")
    B = custom(1, 1, 0, ld, "row")
    C = custom(1, 1, 0, nc, "column-major")
    return Case("vhc_desc", nc, jb, mp, A, B, C, cfg, kernel, reduce, S, conj=(0, 1), **kw)


def pinv_case(n, m, cfg, kernel, reduce, S=1, **kw):
    """svd.cu:749-750: out (n x m) = Vh^H U^H: A = Vh transposed (row-contiguous, conj), B = U (k-contiguous, conj)."""
    A = custom(1, 1, 0, n, "row" if n % 8 == 0 else "row-ragged")
    B = custom(1, n, 0, 1, "k-major")
    C = custom(1, m, 0, 1, "row")
    return Case("pinv", n, m, n, A, B, C, cfg, kernel, reduce, S, conj=(1, 1), **kw)


REPLICAS = [
    left_apply_skip_case(64, 4, 2, 4, 2048, T, WIDE, NONE, streamk=0),
    left_apply_skip_case(64, 4, 2, 4, 2048, ("auto", 0, 0), TINY, NONE),
    left_apply_skip_case(128, 4, 2, 4, 1024, T, WIDE, NONE, streamk=0),
    left_apply_skip_case(256, 4, 2, 4, 1024, T, WIDE, NONE, streamk=1),
    stage2_full_case(64, 4, 4, 4, 16, T, WIDE, NONE, streamk=0),
    stage2_full_case(32, 3, 8, 3, 32, T, WIDE, NONE, streamk=0, beta0=True),
    stage2_full_case(64, 4, 4, 4, 64, ("auto", 0, 0), TINY, NONE),
    stage2_full_case(600, 4, 4, 8, 64, T, TALL, NONE, streamk=0),
    stage2_full_case(40, 4, 4, 8, 1024, T, TALL, NONE, streamk=0, beta0=True),
    stage2_full_case(512, 2, 4, 2, 4096, ("auto", 0, 0), TINY, NONE, chunks=(511, 1)),
    vhc_case(32, 960, 4096, 1024, ("auto", 0, 0), TINY, CLUSTER, 9),
    vhc_case(32, 960, 4096, 1024, ("tma", 1, 0), WIDE, NONE, streamk=1, beta0=True),
    pinv_case(100, 300, ("auto", 0, 0), TINY, CLUSTER, 3, beta0=True),
]

# cp.async grids with 65 536 row tiles (more than gridDim.y holds)
OVER_TALL = [
    Case("over-tall", 2097153, 8, 8, custom(1, 8, 0, 1, "k-major"), custom(1, 1, 0, 8, "row"), custom(1, 8, 0, 1, "row"),
         ("auto", 0, 0), TINY, NONE),
    Case("over-tall", 4194241, 8, 8, custom(1, 8, 0, 1, "k-major"), custom(1, 1, 0, 8, "row"), custom(1, 8, 0, 1, "row"),
         ("small", 0, 0), SMALL, NONE),
    Case("over-tall", 8388481, 8, 8, custom(1, 8, 0, 1, "k-major"), custom(1, 1, 0, 8, "row"), custom(1, 8, 0, 1, "row"),
         ("big", 0, 0), BIG, NONE, beta0=True),
]

ALL_CASES = CASES + REPLICAS + OVER_TALL
COVERAGE = collections.Counter()


# ---- buffers -------------------------------------------------------------------------------------------------------
def _view(buf, op: Op, rows, cols):
    """(rows, cols) strided view of the complex128 buffer `buf` (guard elements excluded) as the descriptor addresses it."""
    return np.lib.stride_tricks.as_strided(buf[FRONT:], shape=(rows // op.inner, op.inner, cols),
                                           strides=(16 * op.s1, 16 * op.s0, 16 * op.sc), writeable=True)


def _extent(op: Op, rows, cols):
    return (rows // op.inner - 1) * op.s1 + (op.inner - 1) * op.s0 + (cols - 1) * op.sc + 1


def poisoned(op: Op, rows, cols, values, off=0):
    """Host buffer holding `values` (rows x cols) where `op` addresses them (plus `off` elements), POISON elsewhere."""
    size = FRONT + off + _extent(op, rows, cols) + BACK
    buf = np.empty(size, np.complex128)
    buf.view(np.uint64)[:] = POISON
    if values is not None:
        _view(buf[off:], op, rows, cols)[...] = values.reshape(-1, op.inner, cols)
    return buf


def values(rng, mode, rows, cols, row_scale=None, col_scale=None):
    if mode == "exact":
        return (rng.integers(-4, 5, (rows, cols)) + 1j * rng.integers(-4, 5, (rows, cols))).astype(np.complex128)
    x = (rng.standard_normal((rows, cols)) + 1j * rng.standard_normal((rows, cols)))
    if row_scale is not None:
        x *= row_scale[:, None]
    if col_scale is not None:
        x *= col_scale[None, :]
    return x


def to_dev(buf):
    return torch.from_numpy(buf.view(np.int64)).to("cuda")


def kernel_names(prof):
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert names, "the profiler recorded no CUDA activity"
    return [n for n in names if "zgemm_" in n or "k_splitk_reduce" in n]


def expected_name(kernel, a_k, b_k):
    kind = "zgemm_tma_kernel<[^<>]*TmaCfg" if kernel in (WIDE, TALL) else "zgemm_dmma_kernel<[^<>]*::Cfg"
    return re.compile(f"{kind}<{CFG_ARGS[kernel]}>, {'true' if a_k else 'false'}, {'true' if b_k else 'false'}>")


TMA_FLAGS = {  # A / B label -> (kmajor, small_inner, swapped) of the tensor map
    "k-major": (1, 0, 0), "row": (0, 0, 0), "r2": (0, 0, 0), "r2-small": (0, 1, 0), "swapped": (1, 0, 1)}


def tma_flags(label):
    if label in TMA_FLAGS:
        return TMA_FLAGS[label]
    if label.startswith("k2-small"):
        return (1, 1, 0)
    assert re.fullmatch(r"k2-\dR", label), label
    return (1, 0, 0)


def run_case(eng, shim, case: Case, seed: int):
    rng = np.random.default_rng(seed)
    M, N, K = case.M, case.N, case.K
    exact = case.mode == "exact"
    alpha, beta = (EXACT_ALPHA, EXACT_BETA) if exact else (GRADED_ALPHA, GRADED_BETA)
    if case.beta0:
        beta = 0.0
    rs = cs = None
    if not exact:
        rs = 2.0 ** rng.integers(-40, 41, M)
        cs = 2.0 ** rng.integers(-40, 41, N)
    A = values(rng, case.mode, M, K, row_scale=rs)
    B = values(rng, case.mode, K, N, col_scale=cs)
    C0 = None if case.beta0 else values(rng, case.mode, M, N, row_scale=rs, col_scale=cs)
    a_off, c_off = case.flags.get("a_off", 0), case.flags.get("c_off", 0)
    hA = poisoned(case.a, M, K, A, a_off)
    hB = poisoned(case.b, N, K, B.T)
    hC = poisoned(case.c, M, N, C0, c_off)
    dA, dB, dC = to_dev(hA), to_dev(hB), to_dev(hC)
    # one call, or heff2_mid's row chunks: chunk i covers rows [r0 * inner, (r0 + n) * inner) of A and C
    calls = []
    if case.chunks:
        r0 = 0
        for n in case.chunks:
            calls.append((n * case.a.inner, r0 * case.a.s1, r0 * case.c.s1))
            r0 += n
    else:
        calls.append((M, 0, 0))
    eng.set_gemm_config(*case.cfg)
    plans, rcs = [], []
    from torch.profiler import ProfilerActivity, profile

    try:
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for m, ao, co in calls:
                desc = (m, N, K, dA.data_ptr() + 16 * (FRONT + a_off + ao), case.a.inner, case.a.s1, case.a.s0, case.a.sc, case.conj[0],
                        dB.data_ptr() + 16 * FRONT, case.b.inner, case.b.s1, case.b.s0, case.b.sc, case.conj[1],
                        dC.data_ptr() + 16 * (FRONT + c_off + co), case.c.inner, case.c.s1, case.c.s0, case.c.sc)
                out = (ctypes.c_longlong * len(PLAN_FIELDS))()
                rcs.append(shim.gemm_desc_run(eng.h, (ctypes.c_longlong * 20)(*desc),
                                              (ctypes.c_double * 4)(alpha.real, alpha.imag, complex(beta).real, complex(beta).imag), out))
                plans.append(dict(zip(PLAN_FIELDS, out)))
            torch.cuda.synchronize()
    finally:
        eng.set_gemm_config("auto", 0, 0)
    assert rcs == [0] * len(calls), (rcs, eng.lib.tdvp_last_error(eng.h))

    # ---- the plan, and the kernel that ran
    names = kernel_names(prof)
    gemm_names = [n for n in names if "zgemm_" in n]
    for p in plans:
        assert (p["kernel"], p["reduce"], p["S"]) == (case.kernel, case.reduce, case.S), p
        if case.streamk is not None:
            assert p["streamk"] == case.streamk, p
        if case.kernel in (WIDE, TALL):
            assert (p["a_kmajor"], p["a_small"], p["a_swapped"]) == tma_flags(case.a.label), (case.a.label, p)
            assert (p["b_kmajor"], p["b_small"], p["b_swapped"]) == tma_flags(case.b.label), (case.b.label, p)
            a_k, b_k = p["a_kmajor"], p["b_kmajor"]
        else:
            a_k, b_k = case.a.sc == 1, case.b.sc == 1
        pat = expected_name(case.kernel, a_k, b_k)
    assert len(gemm_names) == len(calls) and all(pat.search(n) for n in gemm_names), (pat.pattern, names)
    assert sum("k_splitk_reduce" in n for n in names) == (len(calls) if case.reduce == SCRATCH else 0), names

    # ---- guards: A and B untouched, C written exactly where the descriptor addresses it
    outA, outB, outC = (t.cpu().numpy().view(np.complex128) for t in (dA, dB, dC))
    assert np.array_equal(outA.view(np.uint64), hA.view(np.uint64)), "A changed"
    assert np.array_equal(outB.view(np.uint64), hB.view(np.uint64)), "B changed"
    mask = np.zeros(hC.shape[0], bool)
    np.lib.stride_tricks.as_strided(mask[FRONT + c_off:], shape=(M // case.c.inner, case.c.inner, N),
                                    strides=(case.c.s1, case.c.s0, case.c.sc), writeable=True)[...] = True
    words = outC.view(np.uint64).reshape(-1, 2)
    bad = ~mask & np.any(words != POISON, axis=1)
    assert not bad.any(), f"{int(bad.sum())} C elements outside the descriptor were written, first at {np.flatnonzero(bad)[:5]}"
    got = _view(outC[c_off:], case.c, M, N).reshape(M, N)

    # ---- values
    opA = A.conj() if case.conj[0] else A
    opB = B.conj() if case.conj[1] else B
    if exact:
        P = (opA.real @ opB.real - opA.imag @ opB.imag) + 1j * (opA.real @ opB.imag + opA.imag @ opB.real)
        ref = alpha * P + (beta * C0 if C0 is not None else 0)
        np.testing.assert_array_equal(got, ref)
    else:
        ld = np.clongdouble
        ref = ld(alpha) * (opA.astype(ld) @ opB.astype(ld))
        bound = np.abs(alpha) * (np.abs(A) @ np.abs(B))
        if C0 is not None:
            ref = ref + ld(beta) * C0.astype(ld)
            bound = bound + np.abs(beta) * np.abs(C0)
        bound *= 4 * (K + 2) * 2.0 ** -53
        err = np.abs(got.astype(ld) - ref).astype(np.float64)
        assert np.isfinite(got).all()
        worst = np.unravel_index(np.argmax(err / bound), err.shape)
        assert (err <= bound).all(), (worst, err[worst], bound[worst])
    COVERAGE[(KNAME[case.kernel], RNAME[case.reduce] + (str(case.S) if case.S > 1 else ""), case.a.label, case.b.label,
              case.c.label)] += 1


@gpu
@pytest.mark.parametrize("i", range(len(ALL_CASES)), ids=[c.id for c in ALL_CASES])
def test_gemm_path(eng, shim, i):
    run_case(eng, shim, ALL_CASES[i], seed=1000 + i)


# ---- what the case table covers (checked without a GPU) ---------------------------------------------------------------
def _axes(case: Case):
    """-> {axis: value} of one case, the axes of the coverage table in DESIGN.md."""
    kr = f"{KNAME[case.kernel]}/{RNAME[case.reduce]}" + (f"{case.S}" if case.S > 1 else "")
    if case.reduce == CLUSTER:
        kr = f"cluster{case.S}"
    if case.reduce == SCRATCH and case.kernel == TINY:
        kr += f"/cs{case.cfg[2]}"
    if case.kernel == WIDE and case.streamk:
        kr = "tma-wide/stream-K " + ("auto" if case.cfg[0] == "auto" else "forced 4")
    elif case.cfg[0] == "tma_tiles":
        kr = "tma-wide/whole tiles (forced 5)"
    tails = set()
    BM, BN = {BIG: (128, 64), SMALL: (64, 32), TINY: (32, 32), WIDE: (128, 64), TALL: (256, 32)}[case.kernel]
    if case.M in (BM - 1, BM + 1, 148 * BM + 1):
        tails.add("M=BM+-1")
    if case.N in (BN - 1, BN + 1):
        tails.add("N=BN+-1")
    if case.K in (1, 15, 16, 17):
        tails.add(f"K={case.K}")
    if case.S > 1 and case.K % case.S in (1, case.S - 1) or case.K % 8 in (1, 7) and case.S > 1:
        tails.add("K=S*chunk+-1")
    return {"kernel x reduction": {kr}, "A": {case.a.label} | ({"conj"} if case.conj[0] else set()),
            "B": {case.b.label + ("/tall" if case.kernel == TALL else "")} | ({"conj"} if case.conj[1] else set()),
            "C": {case.c.label}, "tails": tails, "c_stream": {f"cs{case.cfg[2]}"} if case.cfg[2] else set(),
            "beta": {"0" if case.beta0 else "nonzero"}}


REQUIRED = {
    "kernel x reduction": {"big/none", "small/none", "tiny/none", "tma-wide/none", "tma-tall/none", "cluster2",
                           "cluster16", "big/scratch4", "tma-wide/scratch2",
                           "tiny/scratch3/cs1", "tma-wide/stream-K auto", "tma-wide/stream-K forced 4",
                           "tma-wide/whole tiles (forced 5)"},
    "A": {"k-major", "row", "row-ragged", "conj", "k2-1R", "k2-2R", "k2-small8", "k2-small32", "k2-small64",
          "k2-small8-desc", "k2-small32-desc", "k2-small64-desc", "swapped", "r2", "r2-small", "untileable96",
          "untileable100"},
    "B": {"k-major", "row", "row-ragged", "conj", "k2-1R", "k2-2R", "k2-small8", "k2-small32", "k2-small8-desc",
          "k2-small32-desc", "swapped", "r2", "r2-small", "untileable96", "untileable100", "k-major/tall", "row/tall",
          "k2-small8/tall", "k2-small16/tall", "k2-small8-desc/tall", "r2-small/tall"},
    "C": {"row", "stage2_full", "left_apply_skip", "column-major"},
    "tails": {"M=BM+-1", "N=BN+-1", "K=1", "K=15", "K=16", "K=17", "K=S*chunk+-1"},
    "c_stream": {"cs1", "cs2"},
    "beta": {"0", "nonzero"},
}


def test_case_table_covers_every_axis_value_twice():
    """Every value of every axis occurs in at least two cases (the GPU cases assert that the plan is the declared one)."""
    seen = collections.defaultdict(collections.Counter)
    for case in ALL_CASES:
        for axis, vals in _axes(case).items():
            seen[axis].update(vals)
    missing = {axis: {v: seen[axis][v] for v in want if seen[axis][v] < 2} for axis, want in REQUIRED.items()}
    assert not any(missing.values()), missing
    assert len({c.id for c in ALL_CASES}) == len(ALL_CASES)


@gpu
def test_coverage_summary():
    """Runs last: the number of cases run for each (kernel, reduction, A geometry, B geometry, C layout)."""
    if not COVERAGE:
        pytest.skip("no GEMM case ran")
    print("\ncases per (kernel, reduction, A, B, C):")
    for key, n in sorted(COVERAGE.items()):
        print(f"  {n:3d}  {' | '.join(key)}")
    print(f"  {sum(COVERAGE.values())} cases in {len(COVERAGE)} combinations")


# ---- K = 0 and leading dimensions (tdvp_zgemm) -----------------------------------------------------------------------
def _zgemm_raw(eng, transA, transB, M, N, K, alpha, beta, A, lda, B, ldb, C, ldc):
    return eng.lib.tdvp_zgemm(eng.h, transA, transB, M, N, K, alpha.real, alpha.imag, ctypes.c_void_p(A.data_ptr()), lda,
                              ctypes.c_void_p(B.data_ptr()), ldb, beta.real, beta.imag, ctypes.c_void_p(C.data_ptr()), ldc)


@gpu
@pytest.mark.parametrize("beta", [0.5 + 1.5j, 0j], ids=["beta", "beta0"])
@pytest.mark.parametrize("M,N,ldc", [(7, 5, 9), (1000, 300, 301)])
def test_zgemm_k0_scales_c(eng, M, N, ldc, beta):
    """K = 0: C = beta C (BLAS), through C's own addressing; with beta = 0 the NaN-poisoned C becomes zeros, and the
    elements between the rows (ldc > N) keep their poison."""
    rng = np.random.default_rng(M + N)
    C0 = values(rng, "exact", M, N)
    hC = poisoned(Op(1, ldc, 0, 1, "row"), M, N, None if beta == 0 else C0)
    dC = to_dev(hC)
    dummy = torch.zeros(4, dtype=torch.complex128, device="cuda")
    base = eng.stats()["launches"]
    assert _zgemm_raw(eng, 0, 0, M, N, 0, 2 - 1j, beta, dummy, 0, dummy, N, dC[2 * FRONT:], ldc) == 0
    torch.cuda.synchronize()
    assert eng.stats()["launches"] > base
    out = dC.cpu().numpy().view(np.complex128)
    got = _view(out, Op(1, ldc, 0, 1, "row"), M, N).reshape(M, N)
    np.testing.assert_array_equal(got, beta * C0 if beta != 0 else np.zeros((M, N)))
    mask = np.zeros(hC.shape[0], bool)
    mask[FRONT:FRONT + M * ldc].reshape(M, ldc)[:, :N] = True
    assert (out.view(np.uint64).reshape(-1, 2)[~mask] == POISON).all()
    assert torch.equal(dummy, torch.zeros_like(dummy))


@gpu
@pytest.mark.parametrize("ta,tb,short", [(0, 0, "lda"), (1, 0, "lda"), (0, 0, "ldb"), (0, 1, "ldb"), (0, 0, "ldc"),
                                         (2, 2, "ldc")])
def test_zgemm_rejects_short_leading_dimension(eng, ta, tb, short):
    """lda / ldb / ldc shorter than the stored row length is TDVP_ERR_ARG, and nothing is launched or written."""
    M, N, K = 40, 24, 16
    lds = {"lda": M if ta else K, "ldb": K if tb else N, "ldc": N}
    lds[short] -= 1
    A, B = (torch.ones(4096, dtype=torch.complex128, device="cuda") for _ in range(2))
    C = torch.full((4096,), 3.0 + 0j, dtype=torch.complex128, device="cuda")
    base = eng.stats()["launches"]
    rc = _zgemm_raw(eng, ta, tb, M, N, K, 1 + 0j, 0j, A, lds["lda"], B, lds["ldb"], C, lds["ldc"])
    assert rc == -1
    assert "leading dimension" in eng.lib.tdvp_last_error(eng.h).decode()
    torch.cuda.synchronize()
    assert eng.stats()["launches"] == base and bool((C == 3.0).all())


@gpu
# ---- contractions through the identity-channel shortcut at tileable D -------------------------------------------------
@pytest.mark.parametrize("cfg", [("auto", 0, 0), ("tma", 0, 0)], ids=["auto", "tma"])
@pytest.mark.parametrize("D,d", [(64, 32), (128, 8)])
def test_heff_identity_shortcut_tileable(eng, D, d, cfg):
    """left_apply_skip / right_apply_skip at D = 64 (small-inner map with descending strides) and D = 128 (swapped map),
    Dl d Dr >= 2^17, against the oracle's einsum contraction."""
    import dataclasses

    from oracle import tdvp_oracle as orc

    rng = np.random.default_rng(D + d)
    w = 4
    psi = values(rng, "graded", D, d * D).reshape(D, d, D)
    L, R = values(rng, "graded", D, w * D).reshape(D, w, D), values(rng, "graded", D, w * D).reshape(D, w, D)
    L[:, 1, :] = np.eye(D)
    R[:, 2, :] = np.eye(D)
    W = values(rng, "graded", w * d, d * w).reshape(w, d, d, w)
    ref = orc.heff_term(L, orc.SiteCore((0, 1, 2), 1, W, False, False), R, psi)
    core = dataclasses.replace(eng.upload_core(W), l_id=1, r_id=2)
    eng.set_gemm_config(*cfg)
    try:
        out = eng.heff_apply([(eng.to_device(L), core, eng.to_device(R), 0.7 - 0.2j)], eng.to_device(psi)).cpu().numpy()
    finally:
        eng.set_gemm_config("auto", 0, 0)
    assert np.abs(out - (0.7 - 0.2j) * ref).max() / np.abs(ref).max() < 1e-12


@gpu
@pytest.mark.parametrize("cfg", [("auto", 0, 0), ("tma", 0, 0)], ids=["auto", "tma"])
def test_keff_identity_shortcut_tileable(eng, cfg):
    """keff_apply with both shortcuts at D = 128 (w = 8: D D w >= 2^17) against the oracle."""
    from oracle import tdvp_oracle as orc

    rng = np.random.default_rng(128)
    D, w = 128, 8
    sig = values(rng, "graded", D, D)
    L, R = values(rng, "graded", D, w * D).reshape(D, w, D), values(rng, "graded", D, w * D).reshape(D, w, D)
    L[:, 3, :] = np.eye(D)
    R[:, 5, :] = np.eye(D)
    ref = orc.keff_term(L, R, sig)
    eng.set_gemm_config(*cfg)
    try:
        out = eng.keff_apply([(eng.to_device(L), eng.to_device(R), 1.0, (3, 5))], eng.to_device(sig)).cpu().numpy()
    finally:
        eng.set_gemm_config("auto", 0, 0)
    assert np.abs(out - ref).max() / np.abs(ref).max() < 1e-12
