"""Two-site TDVP without a GPU: the oracle against exact dynamics, bond growth and truncation, and the product's host sweep
(pytdscf_b200/_twosite.py, Simulator) with the oracle's kernels injected (oracle/two_site_engine.py)."""
import math

import numpy as np
import pytest
import scipy.linalg

import oracle.tdvp_oracle as orc
import oracle.two_site_oracle as tso
from oracle.two_site_engine import TwoSiteOracleEngine
from tests.golden_io import load_run
from tests.two_site_cases import (TRACE_KINDS, complex_mpo_case, dense_hamiltonian, dense_state, oracle_run,
                                  oracle_two_site, product_run, random_canonical_mps, recording_split)


def _exact_case(name):
    return complex_mpo_case() if name == "complex3" else load_run(name)


@pytest.mark.parametrize("name", ["henon_heiles_f2", "exciton_D2", "complex3"])
def test_oracle_two_site_is_exact_at_full_bond_dimension(name):
    """At full bond dimension the two-site projector is the identity: 10 steps equal expm(-iHt) psi0, and the one-site
    oracle, to 1e-10 (Arnoldi at thresh 1e-14, so the Krylov error sits at rounding)."""
    g = _exact_case(name)
    H = dense_hamiltonian(g["operators"], g["dims"], g["coupleJ"])
    assert np.abs(H - H.conj().T).max() < 1e-12
    init = random_canonical_mps(g["dims"], 3)
    dt = 1.0 / np.linalg.norm(H, 2)
    two = oracle_two_site(g, init, bond_dim=None, p_svd=0.0, thresh=1e-14, integrator="arnoldi")
    one = oracle_two_site(g, init, bond_dim=None, p_svd=0.0, thresh=1e-14, integrator="arnoldi")
    for _ in range(10):
        two.propagate_two_site(dt)
        one.propagate(dt)
    ref = scipy.linalg.expm(-1j * H * 10 * dt) @ dense_state(init)
    assert np.abs(dense_state(two.mps) - ref).max() <= 1e-10
    assert np.abs(dense_state(two.mps) - dense_state(one.mps)).max() <= 1e-10


@pytest.mark.parametrize("bond_dim", [4, 8])
def test_bonds_grow_from_a_hartree_product_up_to_the_cap(bond_dim):
    g = load_run("henon_heiles_f6")
    dims = g["dims"]
    hartree = [np.eye(d)[0] for d in dims]
    init = orc.initial_mps(dims, bond_dim, hartree)
    o = oracle_two_site(g, init, bond_dim=bond_dim, p_svd=1e-10, thresh=1e-10, integrator="lanczos")
    caps = [min(bond_dim, math.prod(dims[: p + 1]), math.prod(dims[p + 1:])) for p in range(len(dims) - 1)]
    seen = []
    for _ in range(6):
        o.propagate_two_site(g["dt_au"])
        seen.append(o.bonddim())
        assert all(b <= c for b, c in zip(o.bonddim(), caps, strict=True))
        assert abs(o.norm() - 1.0) < 1e-13
    assert seen[0] != [1] * (len(dims) - 1)        # the product state's bonds of 1 grew in the first step
    assert seen[-1] == [min(c, 4) for c in caps]    # up to the cap within six steps (bond_dim 4), or on the way to it


def test_split_without_norm_conservation_loses_the_discarded_weight():
    rng = np.random.default_rng(5)
    theta = rng.standard_normal((3, 4, 5, 2)) + 1j * rng.standard_normal((3, 4, 5, 2))
    s = np.linalg.svd(theta.reshape(12, 10), compute_uv=False)
    for direction in ("left", "right"):
        for p, cap in ((0.2, 10), (0.0, 4), (1e-12, 10)):
            left, right, s_out, r = tso.split_two_site(theta, direction, p, cap, False)
            cs = np.cumsum(s)
            rp = int(np.nonzero(cs / cs[-1] >= 1 - p)[0][0]) + 1
            assert r == max(1, min(rp, cap))
            kept = np.tensordot(left, right, axes=(2, 0))
            assert abs(np.linalg.norm(kept) ** 2 - np.sum(s[:r] ** 2)) < 1e-12 * np.sum(s**2)
            assert abs((np.linalg.norm(theta) ** 2 - np.linalg.norm(kept) ** 2) - np.sum(s[r:] ** 2)) < 1e-12 * np.sum(s**2)
            _l, _r, _s, r2 = tso.split_two_site(theta, direction, p, cap, True)
            assert abs(np.linalg.norm(np.tensordot(_l, _r, axes=(2, 0))) - np.linalg.norm(theta)) < 1e-12 * np.linalg.norm(theta)


def test_norm_is_conserved_with_conserve_norm_and_leaks_without():
    g = load_run("henon_heiles_f6")
    for cn in (True, False):
        o = oracle_two_site(g, g["init"], bond_dim=2, p_svd=1e-7, thresh=1e-10, integrator="lanczos", conserve_norm=cn)
        for _ in range(3):
            o.propagate_two_site(g["dt_au"])
        if cn:
            assert abs(o.norm() - 1.0) < 1e-13
        else:
            assert o.norm() < 1.0 - 1e-12   # the weight truncated to bond dimension 2 is gone


HOST_CASES = [("henon_heiles_f6", False), ("exciton_D6", False), ("liouville_spin3", False), ("henon_heiles_f6", True)]


@pytest.mark.parametrize("name,merge", HOST_CASES)
def test_host_two_site_logic_reproduces_oracle(name, merge, tmp_path):
    """Simulator.propagate(two_site=True) with the oracle's kernels = TwoSiteOracle.propagate_two_site: identical bond
    dimensions and Krylov traces, observables and the final state to 1e-12 (Lanczos in Hilbert space, Arnoldi in Liouville
    space, and the direct-sum MPO of merge_mpo_terms)."""
    g = load_run(name)
    nstep = 3
    o, rows = oracle_run(g, nstep)
    if merge:
        from pytdscf_b200._mps_cuda import direct_sum_mpo

        n = len(g["dims"])
        assert all(len(k) == n for k in g["operators"])   # every key spans the chain: merge_mpo_terms makes one key
        go = dict(g, operators={tuple((i, i) for i in range(n)): direct_sum_mpo(list(g["operators"].values()))})
        o, rows = oracle_run(go, nstep)
    sim, ener, wf = product_run(g, tmp_path, nstep, eng=TwoSiteOracleEngine(), merge=merge)
    assert [tuple(t) for t in wf.ci_coef.trace] == [(TRACE_KINDS[k], s, n) for k, s, n in o.trace]
    for rec, row in zip(sim.history, rows, strict=True):
        assert rec["bonddim"] == row["bonddim"]
        assert abs(rec["autocorr"] - row["autocorr"]) < 1e-12
        assert abs(rec["norm"] - row["norm"]) < 1e-12
        if g["space"] == "hilbert":
            assert abs(rec["energy"] - row["energy"]) < 1e-12 * max(1.0, abs(row["energy"]))
    assert wf.ci_coef.bonddim() == o.bonddim()
    assert np.abs(dense_state(wf.ci_coef.to_numpy()) - dense_state(o.mps)).max() < 1e-12
    lines = open(f"{g['name']}_2s_prop/bonddim.dat").read().splitlines()
    assert len(lines) == nstep + 1
    assert [[int(b) for b in ln.split()[1:]] for ln in lines[1:]] == [r["bonddim"] for r in rows]


@pytest.mark.parametrize("name", ["exciton_D2", "exciton_D6", "henon_heiles_f2", "henon_heiles_f6", "h2co_D16", "liouville_spin3"])
def test_split_margins_make_identical_ranks_a_fair_device_requirement(name, monkeypatch):
    """Every split of the GPU propagation cases has its cumulative singular-value sums > 1e-10 (relative) away from the cut,
    far beyond the device SVD's rounding, so the device must choose the oracle's ranks."""
    margins = []
    monkeypatch.setattr(tso, "split_two_site", recording_split(1e-7, margins))
    oracle_run(load_run(name), 5, record=False)
    assert margins and min(margins) > 1e-10


def test_two_site_rejects_what_it_does_not_cover(tmp_path):
    import pytdscf_b200 as tb
    from pytdscf_b200._const_cls import RunConfig

    g = load_run("henon_heiles_f2")
    with pytest.raises(NotImplementedError):
        product_run(g, tmp_path, 1, eng=TwoSiteOracleEngine(), adaptive=True)
    with pytest.raises(NotImplementedError):
        product_run(g, tmp_path, 1, eng=TwoSiteOracleEngine(), parallel_split_indices=[(0,), (1,)])
    with pytest.raises(NotImplementedError):
        RunConfig(two_site=True, relax=True)
    model = tb.Model([tb.Exciton(nstate=2)], {"hamiltonian": tb.TensorHamiltonian(
        ndof=1, potential=[[{((0, 0),): tb.TensorOperator(mpo=[np.eye(2).reshape(1, 2, 2, 1)])}]], backend="cuda")}, bond_dim=2)
    sim = tb.Simulator("one", model)
    sim.eng = TwoSiteOracleEngine()
    with pytest.raises(ValueError):
        sim.propagate(maxstep=1, two_site=True, write_files=False)
    with pytest.raises(NotImplementedError):
        sim.relax(maxstep=1, two_site=True, write_files=False)
    with pytest.raises(NotImplementedError):
        sim.operate(two_site=True, write_files=False)
    gate = load_run("gate_exciton_D6")
    from tests.test_gpu_propagation import build_model

    sim = tb.Simulator("gate", build_model(gate))
    sim.eng = TwoSiteOracleEngine()
    with pytest.raises(NotImplementedError):
        sim.propagate(maxstep=1, two_site=True, write_files=False)


def test_two_site_header_and_ctypes_signatures_agree():
    """include/tdvp_b200_two_site.h declares exactly the entry points _lib.SIGNATURES_TWO_SITE binds, tdvp_b200.h includes it,
    and the library exports them (no device needed)."""
    import os
    import re
    import subprocess

    from pytdscf_b200 import _lib

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "tdvp_b200_two_site.h")).read()
    declared = set(re.findall(r"\b(tdvp_[a-z_0-9]+)\s*\(", header)) - set(_lib.SIGNATURES)
    assert declared == set(_lib.SIGNATURES_TWO_SITE)
    assert '#include "tdvp_b200_two_site.h"' in open(os.path.join(root, "include", "tdvp_b200.h")).read()
    lib = _lib.load_library()
    assert all(hasattr(lib, n) for n in declared) and lib.tdvp_abi_version() == 2
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert declared <= set(re.findall(r"\bT (tdvp_[a-z_0-9]+)\b", out))
