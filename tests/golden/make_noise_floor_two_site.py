"""Noise floor of the two-site TDVP oracle (oracle/two_site_oracle.py, TwoSiteOracle.propagate_two_site), in the style of make_noise_floor.py.

For every golden run the two-site oracle is re-run for 5 steps from the golden initial MPS with every one- and two-site
H_eff term output multiplied by (1 + 2e-16 * N(0,1)), one rounding.  The largest change of autocorrelation, energy and
final state over 5 seeds is the floor below which no implementation can be expected to agree with the oracle.  Written
to tests/golden/noise_floor_two_site.json; tests/test_gpu_two_site.py uses max(1e-10, 4 x floor).

    python tests/golden/make_noise_floor_two_site.py
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import oracle.tdvp_oracle as orc  # noqa: E402
import oracle.two_site_oracle as tso  # noqa: E402
from tests.golden_io import RUN_CASES, load_run  # noqa: E402
from tests.two_site_cases import dense_state, oracle_run  # noqa: E402

NSTEP = 5


def run(name, eps, seed):
    rng = np.random.default_rng(seed)
    orig1, orig2 = orc.heff_term, tso.heff2_term
    if eps:
        def noisy1(*a):
            out = orig1(*a)
            return out * (1 + eps * rng.standard_normal(out.shape))

        def noisy2(*a):
            out = orig2(*a)
            return out * (1 + eps * rng.standard_normal(out.shape))
        orc.heff_term, tso.heff2_term = noisy1, noisy2
    try:
        o, rows = oracle_run(load_run(name), NSTEP)
    finally:
        orc.heff_term, tso.heff2_term = orig1, orig2
    return rows, dense_state(o.mps), list(o.trace), o.bonddim()


def main():
    out = {}
    for name in RUN_CASES:
        rows0, st0, tr0, bd0 = run(name, 0.0, 0)
        a = e = s = 0.0
        stable = True
        for seed in range(1, 6):
            rows, st, tr, bd = run(name, 2e-16, seed)
            stable = stable and tr == tr0 and bd == bd0
            a = max(a, max(abs(r["autocorr"] - r0["autocorr"]) for r, r0 in zip(rows, rows0)))
            if rows0[0]["energy"] is not None:
                e = max(e, max(abs(r["energy"] - r0["energy"]) / abs(r0["energy"]) for r, r0 in zip(rows, rows0)))
            s = max(s, float(np.abs(st - st0).max()))
        out[name] = {"autocorr_abs": a, "energy_rel": e, "state_abs": s, "trace_stable": stable}
        print(name, out[name])
    with open(os.path.join(HERE, "noise_floor_two_site.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
