#!/usr/bin/env python
"""Benchmark of the TDVP hot path (BASELINE.json metric: TDVP sweeps/s and H_eff matvec TFLOP/s at D = 256 / 1024).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4|c3|c2|c5|c1] [--impl cuda|reference]

A "step" is one TDVP time step = one forward + one backward half sweep (2 sweeps) of one-site projector-splitting TDVP
over the whole chain (``MPSCoef.propagate``, pytdscf/_mps_cls.py:452-503), properties off.  Default workload: BASELINE
config 4 (radical-pair Liouville-space MPDO, 17 sites, D = 1024, Arnoldi), the configuration the north-star target
(>= 20x the CPU path at D = 1024) is quoted on.

One JSON line (rank 0):
* ``value``     sweeps/s with the MPS, MPO and environments resident in HBM (CUDA events, max over ranks).
* ``e2e``       same metric through the public host-buffer path, >= 5 steps: every step copies the site tensors from pinned
                host memory (H2D), rebuilds the environments, propagates, and copies the tensors + the norm back (D2H).
* ``roofline``  the dominant kernel family (the DMMA ZGEMM): sum of 8*M*N*K over its launches in the timed region / sum of
                their CUDA-event durations on the launching stream, against the measured FP64 DMMA peak.
* ``heff_matvec``  ``tdvp_heff_apply`` alone at D = 256 and D = 1024 (the second half of BASELINE's metric): TFLOP/s
                (algorithmic F_H, SURVEY 8(d)) and fraction of the FP64 tensor peak, CUDA events, best of 5.
* ``d256``      sweeps/s of BASELINE config 3 (LVC pyrazine, 25 sites, D = 256) in the same run.
* ``site_parallel``  BASELINE config 5 (128 sites, D = 512): N = 1 -> the serial algorithm on one GPU; N > 1 -> the
                reference's site-segment-parallel TDVP of ONE chain across the N ranks (NCCL p2p) plus the serial number
                measured on rank 0 in the same run and the strong-scaling efficiency derived from the two.
* ``c1``        BASELINE config 1 (H2CO, D = 16): time per site update and kernel launches per sweep next to the CPU
                reference (the launch-bound regime, SURVEY 8(d)).
* ``cpu_baseline``  (N = 1) the UNMODIFIED reference (oracle/_ref, byte-compiled build product of /root/reference) timed on
                this box's host cores on a bounded sample of the same workload; ``kind`` says "reference" (or "port" when
                only the oracle restatement is available).
* N > 1         the headline workload is "replicas only" in the reference's semantics (SURVEY 8(e): Liouville space is
                excluded from its parallel path): N independent replicas, no data-path collective, weak scaling;
                ``--workload c5`` makes the site-parallel run the headline instead (strong scaling).
``--impl reference`` times the CPU reference alone (rank 0; other ranks exit), see ``run_reference``.
``--dump-outputs DIR`` writes the MPS the timed steps left behind (``dump_outputs``), so that two builds run with the same
arguments can be compared output for output.
"""
from __future__ import annotations

import os
import sys

# The reference arm is BLAS-bound host work.  torchrun exports OMP_NUM_THREADS=1 to every rank unless it is set, which
# would run OpenBLAS single-threaded (r1: the arm timed out at N > 1): give rank 0 all the host cores before NumPy loads.
if "reference" in sys.argv and os.environ.get("RANK", "0") == "0":
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(os.cpu_count() or 1)

import argparse  # noqa: E402
import json  # noqa: E402
import statistics  # noqa: E402
import subprocess  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FP64_DMMA_PEAK_TFLOPS = 37.0  # measured on this pool's B200: profiles/r1_fp64_pipe_microbench.jsonl (64 FMA/clk/SM @1.965 GHz)
PEAK_SOURCE = ("measured FP64 DMMA peak of this pool's B200 (profiles/r1_fp64_pipe_microbench.jsonl; MEASURED_PEAKS.json has "
               "no FP64 entry; cuBLAS ZGEMM 8192^3 = 36.97 TFLOP/s)")
STATS_DIR = os.path.join(ROOT, "bench_stats")
E2E_STEPS = 5
DUMP_BYTES = 60_000_000   # --dump-outputs budget over all files (.npy headers included)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default="c4", choices=["c1", "c2", "c3", "c4", "c5"])
    ap.add_argument("--bond-dim", type=int, default=None, help="override the workload's bond dimension (not a bench line)")
    ap.add_argument("--parallel", default="auto", choices=["auto", "replicas", "sites"],
                    help="N > 1: 'sites' = site-segment-parallel TDVP of ONE chain (strong scaling; default for c5), "
                         "'replicas' = N independent chains (weak scaling; default otherwise)")
    ap.add_argument("--sites", type=int, default=None, help="override the chain length of c5 (not a bench line)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the heff_matvec / d256 / site_parallel / c1 blocks")
    ap.add_argument("--gemm", default="auto", choices=["auto", "big", "small", "tiny", "tma"], help="force a GEMM tile configuration (tuning)")
    ap.add_argument("--no-merge", action="store_true", help="D <= 64 workloads: keep one GEMM chain per MPO key (tuning)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the site tensors after the last timed step as DIR/<name>.npy (float64, <= 60 MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def make_workload(args, name=None):
    from pytdscf_b200 import workloads

    name = name or args.workload
    kw = {}
    if args.bond_dim is not None and name == args.workload:
        kw["D"] = args.bond_dim
    if getattr(args, "sites", None) is not None and name == "c5":
        kw["nsite"] = args.sites
    return workloads.by_name(name, **kw)


def config_dict(wl, world: int, site_parallel: bool, thresh: float = 1e-9) -> dict:
    """The ``config`` entry of the JSON line -- built by ONE function so that both arms emit the same dict."""
    return {"workload": wl.name, "description": wl.description, "sites": len(wl.dims), "bond_dim": wl.bond_dim,
            "integrator": wl.integrator, "dt_au": wl.dt_au, "thresh_sil": thresh,
            "step": "1 time step = 2 half sweeps, properties off",
            "parallelism": "single GPU" if world == 1 else
            (f"site-parallel TDVP, {world} contiguous segments, NCCL p2p of boundary blocks" if site_parallel
             else f"{world} independent replicas (no collective)"),
            "l2": "per-step working set (Krylov basis + contraction intermediates, GBs) >> 126 MB L2; no explicit flush"}


# ----------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows: list[list[str]] = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.rows.append(parts)

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------
# CPU legs
# ----------------------------------------------------------------------------------------------------
def site_shapes(wl):
    from pytdscf_b200._mps_cuda import bond_dims

    return [(bond_dims(wl.dims, i, wl.bond_dim), wl.dims[i]) for i in range(len(wl.dims))]


def blas_threads() -> int:
    try:
        from threadpoolctl import threadpool_info

        return max([int(p.get("num_threads", 1)) for p in threadpool_info()] + [1])
    except Exception:
        return os.cpu_count() or 1


def use_all_cores() -> int:
    """Make the BLAS pools use every host core (explicitly: env defaults differ under torchrun); returns the count in use."""
    n = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_limits

        threadpool_limits(limits=n)
    except Exception:
        pass
    return blas_threads()


def first_full_site(wl) -> int:
    shapes = site_shapes(wl)
    for i, ((dl, dr), _d) in enumerate(shapes):
        if dl == wl.bond_dim and dr == wl.bond_dim:
            return i
    return int(np.argmax([dl * dr for (dl, dr), _ in shapes]))


def reference_sample(wl, budget: str) -> dict:
    """Time the UNMODIFIED reference on ``wl`` (oracle/ref_runner.py).  Workloads whose full time step is affordable on the
    host (estimated < ~40 s) are timed with the reference's own ``MPSCoefMPO.propagate``; the others (config 4, config 5)
    with its own ``propagate_along_sweep`` over the first sites of the chain on the real state -- through the first
    full-bond-dimension site (``budget == "short"``, the ~30 s cpu_baseline leg) or through one site of EVERY distinct
    physical dimension (``budget == "long"``, the reference arm) -- the rest of the sweep being charged per shape class."""
    from oracle import ref_runner as rr

    cores = use_all_cores()
    shapes = site_shapes(wl)
    # algorithmic cost of one sweep in units of D^3-flops, only to choose between the two modes
    est = sum(16.0 * 8 * d * max(dl, dr) ** 2 * min(dl, dr) * 8 for (dl, dr), d in shapes)   # ~ n_H = 8 applies, w ~ 8
    full_ok = est / 3.0e11 < 20.0       # < ~20 s per sweep at ~300 GFLOP/s
    if full_ok:
        nsteps = 2 if budget == "short" else 3
        if wl.bond_dim <= 128 and (os.cpu_count() or 1) > 1:
            # OpenBLAS oversubscription hurts the reference below D ~ 256 (SURVEY 6): give it its best thread count
            from threadpoolctl import threadpool_limits

            best = None
            for c in sorted({1, min(8, os.cpu_count()), os.cpu_count()}):
                with threadpool_limits(limits=c):
                    t = rr.time_bounded_sweep(wl, min(6, len(wl.dims) - 1))["measured_seconds"]
                if best is None or t < best[1]:
                    best = (c, t)
            threadpool_limits(limits=best[0])
            cores = best[0]
        r = rr.time_full_steps(wl, nsteps, warm_steps=1)
        return {"value": r["sweeps_per_s"], "unit": "sweeps/s", "cores": cores, "kind": "reference",
                "sample": (f"unmodified reference (PyTDSCF 1.3.3 NumPy backend, {rr.source_kind()}): MPSCoefMPO.propagate on the "
                           f"whole chain, {nsteps} full time steps after 1 warm-up step (environment bootstrap + einsum "
                           f"expression caching), {r['seconds_per_step']:.2f} s per step"),
                "seconds": r["seconds_per_step"] * nsteps, "seconds_per_step": r["seconds_per_step"]}
    p0 = first_full_site(wl)
    if budget == "short":
        end = p0 + 1
    else:
        seen, end = set(), p0 + 1
        all_d = {d for ((dl, dr), d) in shapes if dl == wl.bond_dim and dr == wl.bond_dim}
        for i in range(p0, len(wl.dims) - 1):
            (dl, dr), d = shapes[i]
            if dl == wl.bond_dim and dr == wl.bond_dim:
                seen.add(d)
                end = i + 1
            if seen == all_d:
                break
    r = rr.time_bounded_sweep(wl, end)
    return {"value": r["sweeps_per_s"], "unit": "sweeps/s", "cores": cores, "kind": "reference",
            "sample": (f"unmodified reference (PyTDSCF 1.3.3 NumPy backend, {rr.source_kind()}): its own "
                       f"propagate_along_sweep(begin_site=0, end_site={end}) on the real state (real Krylov counts), "
                       f"{r['measured_seconds']:.1f} s for the site updates 0..{end - 1}; the remaining {len(r['filled_sites'])} "
                       f"sites of the sweep charged with the measured time of their shape class (flop-scaled where the class "
                       f"was not sampled) -> {r['sweep_seconds_estimate']:.1f} s per sweep"),
            "seconds": r["measured_seconds"], "seconds_per_step": 2.0 * r["sweep_seconds_estimate"],
            "site_seconds": r["site_seconds"], "filled_sites": r["filled_sites"]}


def _herm_block(rng, D, w):
    x = (rng.standard_normal((D, w, D)) + 1j * rng.standard_normal((D, w, D))) / np.sqrt(2 * D)
    return (x + x.conj().transpose(2, 1, 0)) / 2


def port_sample(wl, stats: dict) -> dict:
    """Fallback when the reference build product is absent: one full-D site update of the oracle's NumPy restatement
    (n_H H_eff applies + QR + env update + n_K K_eff applies + absorb on seeded random blocks), extrapolated to sweeps/s
    by algorithmic flops.  ``kind`` = "port"."""
    from oracle import tdvp_oracle as orc

    cores = use_all_cores()
    n_H = max(1, round(stats["avg_matvecs_H"]))
    n_K = max(1, round(stats["avg_matvecs_K"]))
    rng = np.random.default_rng(7)
    p = first_full_site(wl)
    (Dl, Dr), d = site_shapes(wl)[p]
    H = orc.MPOHamiltonian(len(wl.dims), wl.operators, wl.coupleJ)
    psi = rng.standard_normal((Dl, d, Dr)) + 1j * rng.standard_normal((Dl, d, Dr))
    psi /= np.linalg.norm(psi)
    hterms, kterms, flops_H, flops_E, flops_K = {}, {}, 0.0, 0.0, 0.0
    for core in H.calc_point[p]:
        wl_, wr_ = core.data.shape[0], core.data.shape[-1]
        L = _herm_block(rng, Dl, wl_) if not core.is_left else None
        R = _herm_block(rng, Dr, wr_) if not core.is_right else None
        hterms[core.key] = (L, core, R)
        mid = 8.0 * Dl * Dr * (d * d if core.data.ndim == 4 else d) * wl_ * wr_
        if L is not None:
            flops_H += 8.0 * Dl * Dl * Dr * d * wl_
            flops_E += 8.0 * Dl * Dl * Dr * d * wl_
        flops_H += mid
        flops_E += mid + 8.0 * Dl * Dr * Dr * d * wr_
        if R is not None:
            flops_H += 8.0 * Dl * Dr * Dr * d * wr_
            kterms[core.key] = (_herm_block(rng, Dr, wr_), R)
            flops_K += 16.0 * wr_ * Dr**3
    t0 = time.perf_counter()
    x = psi
    for _ in range(n_H):
        x = orc.heff_apply(hterms, 0.0, x)
        x /= np.linalg.norm(x)
    A, sigma = orc.shift_qr(x)
    for _key, (L, core, _R) in hterms.items():
        orc.env_update_term("A", A, A, L, core)
    s = sigma
    for _ in range(n_K):
        if kterms:
            s = orc.keff_apply(kterms, 0.0, s)
            s /= np.linalg.norm(s)
    np.tensordot(s, psi, axes=(1, 0))
    sec = time.perf_counter() - t0
    rate = (n_H * flops_H + flops_E + n_K * flops_K) / sec
    return {"value": rate / stats["flops_per_sweep"], "unit": "sweeps/s", "cores": cores, "kind": "port",
            "sample": (f"oracle restatement (oracle/_ref not built): one site update at site {p} (Dl={Dl}, d={d}, Dr={Dr}), {n_H} H_eff "
                       f"applies + QR + env update + {n_K} K_eff applies + absorb on seeded random blocks, {sec:.2f} s, extrapolated "
                       f"with {stats['flops_per_sweep'] / 1e12:.3f} TFLOP/sweep"),
            "seconds": sec, "seconds_per_step": 2.0 * stats["flops_per_sweep"] / rate}


def load_stats(wl_name: str) -> dict | None:
    path = os.path.join(STATS_DIR, wl_name + ".json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return None


def default_stats(wl) -> dict:
    """Analytic stand-in (only for the ``port`` fallback on workloads without recorded Krylov counts)."""
    n_H, n_K = 7.0, 4.0
    flops = 0.0
    for p, ((Dl, Dr), d) in enumerate(site_shapes(wl)):
        fH = 16.0 * 8 * d * Dl * Dr * max(Dl, Dr)
        flops += (n_H + 1) * fH + n_K * 16.0 * 8 * Dr**3
    return {"avg_matvecs_H": n_H, "avg_matvecs_K": n_K, "flops_per_sweep": flops, "source": "analytic default"}


def cpu_baseline(wl, stats: dict | None, budget: str = "short") -> dict:
    from oracle import ref_runner as rr

    if rr.source_kind() is not None:
        return reference_sample(wl, budget)
    return port_sample(wl, stats or load_stats(wl.name) or default_stats(wl))


# ----------------------------------------------------------------------------------------------------
def run_reference(args):
    """``--impl reference``: the unmodified reference on the box's host cores, rank 0 only.  One sample of the bounded
    workload is the "step"; it is measured ONCE (a second pass would repeat identical BLAS calls for minutes) and the line
    says so (``samples_timed``).  ``extrapolation_check`` validates the shape-class extrapolation on config 3, where a full
    step of the reference is affordable: its own full MPSCoefMPO.propagate step against the bounded-sweep estimate."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_runner as rr

    wl = make_workload(args)
    t_start = time.perf_counter()
    cb = cpu_baseline(wl, None, budget="long")
    check = None
    # (N = 1 line only: the check costs ~70 s of host time and would say the same thing in every --gpus N line)
    if rr.source_kind() is not None and args.workload == "c4" and int(os.environ.get("WORLD_SIZE", "1")) == 1:
        w3 = make_workload(args, "c3")
        full = rr.time_full_steps(w3, 2, warm_steps=1)
        p0 = first_full_site(w3)
        bounded = rr.time_bounded_sweep(w3, p0 + 2)
        check = {"workload": w3.name, "full_step_sweeps_per_s": full["sweeps_per_s"],
                 "bounded_sweep_estimate_sweeps_per_s": bounded["sweeps_per_s"],
                 "estimate_over_measured": bounded["sweeps_per_s"] / full["sweeps_per_s"],
                 "note": "the reference's own full time step (2 steps after 1 warm-up) vs the shape-class estimate from "
                         f"propagate_along_sweep over sites 0..{p0 + 1}; the same estimator produces the headline value"}
    world = int(os.environ.get("WORLD_SIZE", "1"))
    site_parallel = world > 1 and (args.parallel == "sites" or (args.parallel == "auto" and args.workload == "c5"))
    out = {"impl": "reference", "metric": "tdvp_sweeps_per_sec", "value": cb["value"], "unit": "sweeps/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "samples_timed": 1, "ms_per_step": cb["seconds_per_step"] * 1e3,
           "higher_is_better": True, "scaling": "strong" if site_parallel else "weak", "vs_baseline": None,
           "dtype": "complex128", "data": "synthetic", "config": config_dict(wl, world, site_parallel),
           "cpu_baseline": cb, "wall_s": time.perf_counter() - t_start,
           "e2e": {"value": cb["value"], "unit": "sweeps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if check is not None:
        out["extrapolation_check"] = check
    print(json.dumps(out))


# ----------------------------------------------------------------------------------------------------
# GPU measurement of one workload
# ----------------------------------------------------------------------------------------------------
class Bench:
    def __init__(self, args):
        import torch

        from pytdscf_b200 import parallel
        from pytdscf_b200._engine import Engine

        self.torch = torch
        self.args = args
        # TDVP_BENCH_BACKEND=gloo (debugging only, never a bench line): lets more ranks than GPUs share the devices
        backend = os.environ.get("TDVP_BENCH_BACKEND", "nccl")
        dev = int(os.environ.get("LOCAL_RANK", "0")) % max(1, torch.cuda.device_count())
        torch.cuda.set_device(dev)
        self.info = parallel.init_from_env(backend)
        self.rank, self.world, self.local_rank, self.dist = self.info.rank, self.info.world, dev, self.info.dist
        self.eng = Engine(dev)
        if args.gemm != "auto":
            self.eng.set_gemm_config(args.gemm, 0, 0)

    def barrier(self, group: bool = True):
        self.torch.cuda.synchronize()
        if self.dist is not None and group:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def build(self, wl, site_parallel: bool):
        from pytdscf_b200._const_cls import RunConfig
        from pytdscf_b200._mps_cuda import DeviceMPO, MPSCoefCuda

        model = wl.model()
        # launch-bound workloads (D <= 64) run the whole-chain MPO keys as one direct-sum MPO (DeviceMPO.merge_terms)
        merge = wl.bond_dim <= 64 and not site_parallel and not self.args.no_merge
        H = DeviceMPO(self.eng, model.hamiltonian, merge_terms=merge)
        self.last_merged = bool(H.merged)
        cfg = RunConfig(jobname="bench", space=wl.space, integrator=wl.integrator, conserve_norm=wl.conserve_norm)
        if site_parallel:
            from pytdscf_b200._mps_parallel import Comm, MPSCoefParallelCuda, balanced_split

            # contiguous segments of equal SWEEP COST (the end sites of a chain have small bonds and are nearly free); the
            # reference takes the split from the user (parallel_split_indices), this is the choice a user would make
            split = balanced_split(wl.dims, wl.bond_dim, self.world)
            self.last_split = split
            mps = MPSCoefParallelCuda.distribute(self.eng, Comm(self.info, self.eng.torch_device), model, split)
        else:
            mps = MPSCoefCuda.alloc_random(self.eng, model)
        return mps, H, cfg

    def measure(self, wl, steps: int, warmup: int, *, site_parallel: bool = False, collective: bool = True,
                sample_clocks: bool = False, dump_dir: str | None = None) -> dict:
        """W warm-up steps, then exactly K timed steps between barrier + synchronize, CUDA events, max over ranks.
        ``collective`` False: this rank measures alone (no barrier / reduction with the other ranks).  ``dump_dir``: the
        MPS after the last timed step goes there (``dump_outputs``), before any untimed pass moves it on."""
        torch, eng, dist = self.torch, self.eng, (self.dist if collective else None)
        mps, H, cfg = self.build(wl, site_parallel)
        dt = wl.dt_au
        us_per_launch = 1e9
        for iw in range(warmup):
            if iw == warmup - 1:
                torch.cuda.synchronize()
                l0, t0 = eng.stats()["launches"], time.perf_counter()
            mps.propagate(dt, H, cfg)
            if iw == warmup - 1:
                torch.cuda.synchronize()
                us_per_launch = (time.perf_counter() - t0) * 1e6 / max(1, eng.stats()["launches"] - l0)
        self.barrier(collective)
        # Per-launch CUDA events (roofline) ride inside the timed region when the step is GPU-bound (>= 40 us of step time
        # per launch: two event records per launch are < 1 % there) and move to a separate pass of the same K steps when
        # the stream is launch-bound (D <= 64 workloads), where they would cost ~15 % of the reported time.
        in_region = us_per_launch >= 40.0
        if dist is not None:
            flag = torch.tensor([1.0 if in_region else 0.0], device="cuda", dtype=torch.float64)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            in_region = bool(flag.item() > 0.5)
        sampler = ClockSampler(self.local_rank) if sample_clocks else None
        if sampler:
            sampler.start()
        eng.reset_stats()
        if in_region:
            eng.gemm_profile(True, reset=True)
        launches0 = eng.stats()["launches"]
        mps.record_trace = True
        mps.trace = []
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier(collective)
        ev0.record()
        for _ in range(steps):
            mps.propagate(dt, H, cfg)
        ev1.record()
        self.barrier(collective)
        ms = ev0.elapsed_time(ev1)
        clocks = sampler.stop() if sampler else None
        if dump_dir is not None:
            dump_outputs(mps, dump_dir, prefix="" if self.world == 1 else f"rank{self.rank}_", budget=DUMP_BYTES // self.world)
        ms_prof = ms
        if in_region:
            prof = eng.gemm_profile(False)
            breakdown = eng.profile_breakdown()
        st = eng.stats()
        launches = st["launches"] - launches0
        trace = np.array(mps.trace)
        mps.record_trace = False
        if not in_region:
            # launch-bound workloads only: profiled pass (NOT the reported time) of the same K steps
            eng.gemm_profile(True, reset=True)
            pv0, pv1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            self.barrier(collective)
            pv0.record()
            for _ in range(steps):
                mps.propagate(dt, H, cfg)
            pv1.record()
            self.barrier(collective)
            ms_prof = pv0.elapsed_time(pv1)
            prof = eng.gemm_profile(False)
            breakdown = eng.profile_breakdown()
        if dist is not None:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        flops_all = st["flops"]
        if site_parallel and dist is not None:
            t = torch.tensor([flops_all], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            flops_all = float(t.item())
        nH = trace[trace[:, 0] == 0][:, 2] if len(trace) else np.array([0.0])
        nK = trace[trace[:, 0] == 1][:, 2] if len(trace) else np.array([0.0])
        gemm_tflops = prof["flops"] / (prof["ms"] * 1e-3) / 1e12 if prof["ms"] > 0 else 0.0
        top = sorted(breakdown.items(), key=lambda kv: -kv[1]["ms"])
        return {"mps": mps, "H": H, "cfg": cfg, "merged": bool(getattr(H, "merged", False)), "ms": ms, "ms_prof": ms_prof, "steps": steps, "clocks": clocks, "launches": int(launches),
                "trace_len": len(trace), "flops_all": flops_all,
                "avg_matvecs_H": float(nH.mean()), "avg_matvecs_K": float(nK.mean()) if len(nK) else 0.0,
                "gemm_tflops": gemm_tflops, "gemm_launches": int(prof["launches"]), "gemm_share": prof["ms"] / ms_prof,
                "in_region": in_region, "us_per_launch": us_per_launch,
                "breakdown_top": {k: {"share": round(v["ms"] / ms_prof, 4), "launches": v["launches"],
                                      "tflops": round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 2) if v["ms"] > 0 and v["flops"] > 0 else None}
                                  for k, v in top[:12]}}

    # -- e2e: host buffers in, host buffers out, every step --------------------------------------------
    def e2e(self, wl, m: dict, site_parallel: bool) -> dict:
        torch, eng, dist = self.torch, self.eng, self.dist
        from pytdscf_b200._mps_cuda import MPSCoefCuda

        mps, H, cfg, dt = m["mps"], m["H"], m["cfg"], wl.dt_au
        if site_parallel:
            # segment state (site tensors, both saved gauges, boundary bond matrices) lives in pinned host memory between
            # steps; the environment blocks are caches derived from it and stay on the device
            def state_refs():
                refs = [(sc, "data") for grp in (mps.sites, mps.superblock_all_A, mps.superblock_all_B) for sc in grp]
                if mps.joint_sigvec is not None:
                    refs += [(mps, "joint_sigvec"), (mps, "joint_sigvec_not_pinv")]
                return refs

            host = [torch.empty(getattr(o, a).shape, dtype=torch.complex128).pin_memory() for o, a in state_refs()]
            for hb, (o, a) in zip(host, state_refs(), strict=True):
                hb.copy_(getattr(o, a))
            nbytes = sum(hb.numel() * 16 for hb in host)

            def step():
                for hb, (o, a) in zip(host, state_refs(), strict=True):
                    setattr(o, a, hb.to(eng.torch_device, non_blocking=True))
                mps.propagate(dt, H, cfg)
                refs = state_refs()
                if len(refs) != len(host) or any(getattr(o, a).shape != hb.shape for hb, (o, a) in zip(host, refs)):
                    raise RuntimeError("segment state changed shape during a step")
                for hb, (o, a) in zip(host, refs, strict=True):
                    hb.copy_(getattr(o, a), non_blocking=True)

            path = "pinned host segment state -> H2D -> MPSCoefParallelCuda.propagate -> D2H, every rank"
            d2h_extra, jobs = 0, 1
        else:
            host = [torch.empty(s.data.shape, dtype=torch.complex128).pin_memory() for s in mps.sites]
            for hbuf, s in zip(host, mps.sites, strict=True):
                hbuf.copy_(s.data)
            gauges = [s.gauge for s in mps.sites]
            nbytes = sum(hb.numel() * 16 for hb in host)
            norm_host = torch.empty(1, dtype=torch.float64).pin_memory()

            def step():
                cores = [hb.to(eng.torch_device, non_blocking=True) for hb in host]
                m2 = MPSCoefCuda(eng, cores, gauges)  # fresh object: environments are rebuilt from scratch
                m2.niter_krylov = dict(mps.niter_krylov)
                m2.propagate(dt, H, cfg)
                for hb, s in zip(host, m2.sites, strict=True):
                    hb.copy_(s.data, non_blocking=True)
                norm_host.copy_(torch.linalg.vector_norm(m2.sites[0].data).reshape(1), non_blocking=True)
                mps.niter_krylov = m2.niter_krylov

            path = "pinned host MPS -> H2D -> MPSCoefCuda.propagate (environments rebuilt) -> D2H of MPS + norm"
            d2h_extra, jobs = 8, self.world
        step()   # untimed: first use of the pinned buffers / torch's norm kernel initialises lazily
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(E2E_STEPS):
            step()
        e1.record()
        self.barrier()
        ems = e0.elapsed_time(e1)
        tot = nbytes
        if dist is not None:
            t = torch.tensor([ems, float(nbytes)], device="cuda", dtype=torch.float64)
            dist.all_reduce(t[:1], op=dist.ReduceOp.MAX)
            if site_parallel:
                dist.all_reduce(t[1:], op=dist.ReduceOp.SUM)
            ems, tot = float(t[0].item()), int(t[1].item())
        return {"value": 2 * E2E_STEPS * jobs / (ems * 1e-3), "unit": "sweeps/s", "h2d_bytes_per_step": tot,
                "d2h_bytes_per_step": tot + d2h_extra, "steps": E2E_STEPS, "path": path}

    # -- H_eff matvec alone (second half of the BASELINE metric) -----------------------------------------
    def heff_matvec(self) -> list:
        torch, eng = self.torch, self.eng
        g = torch.Generator(device="cuda").manual_seed(7)

        def rnd(*shape):
            return torch.view_as_complex(torch.randn(*shape, 2, dtype=torch.float64, device="cuda", generator=g))

        rows = []
        for label, D, d, w in (("D=256 (config-3 site: d=10, w=6)", 256, 10, 6), ("D=1024 (config-4 site: d=4, w=8)", 1024, 4, 8)):
            psi, L, R = rnd(D, d, D), rnd(D, w, D), rnd(D, w, D)
            core = eng.upload_core(rnd(w, d, d, w).cpu().numpy())
            terms = [(L, core, R, 1.0)]
            fH = 8.0 * (2.0 * D * D * D * d * w + D * D * d * d * w * w)
            for _ in range(2):
                eng.heff_apply(terms, psi)
            torch.cuda.synchronize()
            best = 1e30
            for _ in range(5):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                eng.heff_apply(terms, psi)
                e1.record()
                torch.cuda.synchronize()
                best = min(best, e0.elapsed_time(e1))
            tf = fH / (best * 1e-3) / 1e12
            rows.append({"case": label, "D": D, "d": d, "w": w, "ms": round(best, 4), "tflops": round(tf, 2),
                         "frac_of_fp64_peak": round(tf / FP64_DMMA_PEAK_TFLOPS, 3)})
            del psi, L, R
        return rows


def dump_outputs(mps, out_dir: str, prefix: str = "", budget: int = DUMP_BYTES) -> None:
    """Write every site tensor of ``mps`` (what a caller of ``propagate`` receives) as ``out_dir/<prefix>site<i>.npy``:
    complex128 stored as float64 (real, imag) pairs in a trailing axis of 2.  When the whole chain exceeds ``budget`` bytes,
    each site tensor larger than an equal share of it is replaced by the flat elements at a fixed, seeded set of sorted
    indices, shape (k, 2): the same elements in every run with the same arguments."""
    import torch

    sites = [s.data for s in mps.sites]
    cap = None
    if sum(t.numel() for t in sites) * 16 + 128 * len(sites) > budget:
        cap = (budget // len(sites) - 128) // 16
    os.makedirs(out_dir, exist_ok=True)
    for i, t in enumerate(sites):
        t = t.detach()
        n = t.numel()
        if cap is not None and n > cap:
            idx = np.sort(np.random.default_rng([2024, i]).choice(n, cap, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, f"{prefix}site{i:03d}.npy"), torch.view_as_real(t.resolve_conj().contiguous()).cpu().numpy())


def summarize(wl, m: dict, world: int, site_parallel: bool) -> dict:
    jobs = 1 if site_parallel else world
    return {"workload": wl.name, "sweeps_per_s": 2 * m["steps"] * jobs / (m["ms"] * 1e-3), "ms_per_step": m["ms"] / m["steps"],
            "steps": m["steps"], "gpu_launches": m["launches"], "gemm_tflops": round(m["gemm_tflops"], 2),
            "gemm_frac_of_fp64_peak": round(m["gemm_tflops"] / FP64_DMMA_PEAK_TFLOPS, 3), "gemm_share_of_step": round(m["gemm_share"], 4),
            "avg_matvecs_H": m["avg_matvecs_H"], "avg_matvecs_K": m["avg_matvecs_K"]}


def run_cuda(args):
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl cuda needs a CUDA device (no CPU fallback)")
    b = Bench(args)
    rank, world, dist, eng = b.rank, b.world, b.dist, b.eng
    wl = make_workload(args)
    site_parallel = world > 1 and (args.parallel == "sites" or (args.parallel == "auto" and args.workload == "c5"))

    m = b.measure(wl, args.steps, args.warmup, site_parallel=site_parallel, sample_clocks=True, dump_dir=args.dump_outputs)
    jobs = 1 if site_parallel else world
    value = 2 * args.steps * jobs / (m["ms"] * 1e-3)
    flops_per_sweep = m["flops_all"] / (2 * args.steps)
    stats = {"avg_matvecs_H": m["avg_matvecs_H"], "avg_matvecs_K": m["avg_matvecs_K"], "flops_per_sweep": flops_per_sweep,
             "source": "bench.py GPU run"}
    e2e = None if args.no_e2e else b.e2e(wl, m, site_parallel)
    for k in ("mps", "H", "cfg"):
        m.pop(k, None)
    torch.cuda.empty_cache()

    extras: dict = {}
    if not args.no_extras and args.workload == "c4" and args.bond_dim is None:
        if rank == 0:
            extras["heff_matvec"] = b.heff_matvec()
        # D = 256 half of the metric: config 3 on this rank alone (no collective), same run
        if rank == 0:
            w3 = make_workload(args, "c3")
            m3 = b.measure(w3, 3, 2, collective=False)
            extras["d256"] = summarize(w3, m3, 1, False)
            del m3
            w1 = make_workload(args, "c1")
            m1 = b.measure(w1, 10, 3, collective=False)
            n1 = len(w1.dims)
            extras["c1"] = {"workload": w1.name, "sweeps_per_s": 2 * 10 / (m1["ms"] * 1e-3),
                            "us_per_site_update": m1["ms"] * 1e3 / (10 * 2 * n1), "launches_per_sweep": m1["launches"] / 20,
                            "mpo_direct_sum": m1["merged"]}
            del m1
            torch.cuda.empty_cache()
        b.barrier()
        # config 5 (128 sites, D = 512): serial on one GPU (rank 0 alone); N > 1: + the site-parallel run over all ranks
        w5 = make_workload(args, "c5")
        sp: dict = {"workload": w5.name}
        if rank == 0:
            ms5 = b.measure(w5, 1, 1, collective=False)
            sp["serial_1gpu"] = summarize(w5, ms5, 1, False)
            del ms5
            torch.cuda.empty_cache()
        b.barrier()
        if world > 1:
            mp5 = b.measure(w5, 2, 1, site_parallel=True)
            if rank == 0:
                sp["parallel"] = summarize(w5, mp5, world, True)
                sp["parallel"]["segments"] = world
                sp["parallel"]["first_site_of_segment"] = list(getattr(b, "last_split", []))
                sp["strong_scaling_efficiency"] = sp["parallel"]["sweeps_per_s"] / (world * sp["serial_1gpu"]["sweeps_per_s"])
                sp["speedup_over_1gpu_serial"] = sp["parallel"]["sweeps_per_s"] / sp["serial_1gpu"]["sweeps_per_s"]
                sp["breakdown_top"] = mp5["breakdown_top"]
                sp["note"] = ("one chain, contiguous site segments, even/odd counter-sweeps + joint boundary update (reference "
                              "MPSCoefParallel, _mps_parallel.py:106-268), NCCL p2p; efficiency = parallel / (N x serial 1-GPU run of "
                              "the same workload measured on rank 0 in this process)")
            del mp5
        extras["site_parallel"] = sp

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    ncu = None
    ncu_path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(ncu_path):
        with open(ncu_path) as f:
            ncu = json.load(f).get(wl.name)
    out = {
        "metric": "tdvp_sweeps_per_sec", "value": value, "unit": "sweeps/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": m["ms"] / args.steps, "higher_is_better": True,
        "scaling": "strong" if site_parallel else "weak",
        "vs_baseline": None, "dtype": "complex128", "data": "synthetic",
        "config": config_dict(wl, world, site_parallel),
        "clocks": m["clocks"],
        "heff_tflops": m["flops_all"] / (m["ms"] * 1e-3) / 1e12,
        "heff_tflops_note": "algorithmic H_eff + K_eff + env-update flops of the reference's contraction (SURVEY 8(d) formula, identity "
                            "MPO channels included) / wall time of the timed region (all kernels); the roofline entry counts "
                            "the flops the GEMM launches actually execute",
        "krylov": {"avg_matvecs_H": m["avg_matvecs_H"], "avg_matvecs_K": m["avg_matvecs_K"],
                   "solves_per_step": m["trace_len"] / args.steps, "tflop_per_sweep": flops_per_sweep / 1e12},
        "gpu_launches": m["launches"],
        "mpo_direct_sum": bool(m.get("merged", False)),
        "roofline": {"kernel": "zgemm (DMMA)", "bound": "tensor", "achieved": m["gemm_tflops"], "peak": FP64_DMMA_PEAK_TFLOPS,
                     "unit": "TFLOP/s", "frac": m["gemm_tflops"] / FP64_DMMA_PEAK_TFLOPS,
                     "traffic": None if ncu is None else ncu.get("dram_bytes_per_launch"),
                     "launches": m["gemm_launches"], "share_of_step": m["gemm_share"],
                     "measured_in": "the timed region" if m["in_region"] else
                     f"separate profiled pass of the same {args.steps} steps ({m['ms_prof'] / args.steps:.1f} ms/step with per-launch "
                     f"events; the step is launch-bound at {m['us_per_launch']:.0f} us per launch)",
                     "peak_source": PEAK_SOURCE},
        "breakdown_top": m["breakdown_top"],
    }
    out.update(extras)
    if e2e is not None:
        out["e2e"] = e2e
    if world == 1 and not args.no_cpu_baseline:
        try:
            out["cpu_baseline"] = cpu_baseline(wl, stats, budget="short")
        except Exception as exc:  # a broken reference build product must not take the GPU line down: fall back to the port
            out["cpu_baseline"] = port_sample(wl, stats)
            out["cpu_baseline"]["reference_error"] = repr(exc)
        if "c1" in extras:
            try:
                from oracle import ref_runner as rr

                if rr.source_kind() is not None:
                    # D = 16: BLAS threading overhead dominates the reference (SURVEY 6 / 8(d)), so it gets its best of
                    # {1, 8, all} threads -- the launch-bound regime is where the CPU could win and must not be handicapped
                    from threadpoolctl import threadpool_limits

                    ncpu = os.cpu_count() or 1
                    w1 = make_workload(args, "c1")
                    by_threads = {}
                    for c in sorted({1, min(8, ncpu), ncpu}):
                        with threadpool_limits(limits=c):
                            by_threads[c] = rr.time_full_steps(w1, 5, warm_steps=1)
                    best = max(by_threads, key=lambda c: by_threads[c]["sweeps_per_s"])
                    r1 = by_threads[best]
                    extras["c1"]["cpu_reference_sweeps_per_s"] = r1["sweeps_per_s"]
                    extras["c1"]["cpu_reference_us_per_site_update"] = r1["seconds_per_step"] * 1e6 / (2 * len(w1.dims))
                    extras["c1"]["cpu_reference_threads"] = best
                    extras["c1"]["cpu_reference_sweeps_per_s_by_threads"] = {str(c): round(v["sweeps_per_s"], 3) for c, v in by_threads.items()}
                    out["c1"] = extras["c1"]
            except Exception as exc:  # the CPU leg must never take the GPU line down
                out["c1"]["cpu_reference_error"] = repr(exc)
    print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
