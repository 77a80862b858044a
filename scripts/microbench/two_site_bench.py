"""Two-site TDVP on the B200: tdvp_heff2_apply throughput, tdvp_split2 latency and one two-site time step with its
per-label breakdown.  JSON lines to the file given as the first argument (default profiles/two_site_bench.jsonl).

  heff2: one full-core MPO term (L, W1, W2, R) per call at a config-3 pair (D = 256, d1 = d2 = 10, w = 6) and a config-4
         pair (D = 1024, d = 4, w = 8); CUDA events, best of 5; flops F_H2 = 8 (Dl^2 d1 d2 Dr wl + Dl Dr d1^2 d2 wl wm +
         Dl Dr d1 d2^2 wm wr + Dl d1 d2 Dr^2 wr).
  split2: Jacobi-SVD split of a random (Dl d1) x (d2 Dr) matricisation, m = n = 256, 512, 1024, 2560 (d1 = d2 = 4).
  step:   one Simulator two-site time step of a config-2-shaped chain (Henon-Heiles, f = 64, N = 8, D = 64) after one
          warm-up step; total wall time and the per-label breakdown of the step, with the share of the split.

    python scripts/microbench/two_site_bench.py [out.jsonl]
"""
import json
import os
import subprocess
import sys
import tempfile
import time

import torch

sys.path.insert(0, ".")
from pytdscf_b200._engine import Engine  # noqa: E402


def timeit(fn, reps=5):
    fn()
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best


def gpu_info() -> dict:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception:     # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown"}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "two_site_bench.jsonl")
    info = gpu_info()
    eng = Engine(0)
    g = torch.Generator(device="cuda").manual_seed(7)

    def rnd(*shape):
        return torch.randn(shape, dtype=torch.complex128, device="cuda", generator=g)

    lines = []
    for label, D, d, w in [("config 3 pair (D=256, d=10, w=6)", 256, 10, 6), ("config 4 pair (D=1024, d=4, w=8)", 1024, 4, 8)]:
        theta, L, R = rnd(D, d, d, D), rnd(D, w, D), rnd(D, w, D)
        W1, W2 = eng.upload_core(rnd(w, d, d, w).cpu().numpy()), eng.upload_core(rnd(w, d, d, w).cpu().numpy())
        terms = [(L, W1, W2, R, 1.0)]
        ms = timeit(lambda: eng.heff2_apply(terms, theta))
        n = D * d * d * D
        fl = 8.0 * (n * D * w + n * d * w * w + n * d * w * w + n * D * w)
        lines.append({"bench": "heff2_apply", "case": label, "ms": ms, "flops": fl, "tflops": fl / ms / 1e9, **info})
        del theta, L, R, W1, W2
        torch.cuda.empty_cache()
    for m in (256, 512, 1024, 2560):
        Dl = m // 4
        theta = rnd(Dl, 4, 4, Dl)
        reps = 5 if m <= 1024 else 2
        ms = timeit(lambda: eng.split2("right", theta, 1e-7, m, True), reps=reps)
        lines.append({"bench": "split2", "m": m, "n": m, "ms": ms, **info})

    import pytdscf_b200 as tb
    from pytdscf_b200.workloads import by_name

    wl = by_name("c2")
    model = wl.model()
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        os.chdir(tmp)
        try:
            sim = tb.Simulator("c2_two_site", model, verbose=0)
            sim.eng = eng
            _, wf = sim.propagate(stepsize=wl.dt_fs, maxstep=3, two_site=True, energy=False, autocorr=False, norm=False,
                                  populations=False, write_files=False)
            ham = wf.device_op(model.hamiltonian)
            torch.cuda.synchronize()
            eng.gemm_profile(True, reset=True)
            t0 = time.perf_counter()
            wf.ci_coef.propagate(wl.dt_fs / tb.units.au_in_fs, ham, sim.cfg)
            torch.cuda.synchronize()
            sec = time.perf_counter() - t0
            eng.gemm_profile(False)
            prof = eng.profile_breakdown()
        finally:
            os.chdir(cwd)
    labels = prof.get("labels", prof)
    split_ms = sum(v.get("ms", 0.0) for k, v in labels.items() if isinstance(v, dict) and k.startswith("svd."))
    total_ms = sum(v.get("ms", 0.0) for k, v in labels.items() if isinstance(v, dict))
    lines.append({"bench": "two_site_step", "case": wl.name, "bonddim_max": max(wf.ci_coef.bonddim()), "step_s": sec,
                  "device_ms_profiled": total_ms, "split_ms": split_ms,
                  "split_share_of_profiled": split_ms / total_ms if total_ms else None, "breakdown": labels, **info})
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")
    for ln in lines:
        print(json.dumps({k: v for k, v in ln.items() if k != "breakdown"}))


if __name__ == "__main__":
    main()
