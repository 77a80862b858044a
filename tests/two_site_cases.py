"""Shared cases of the two-site TDVP tests (tests/test_two_site_cpu.py, tests/test_gpu_two_site.py): dense Hamiltonians of
small chains, random canonical MPS, oracle runs, and Simulator runs of the product."""
from __future__ import annotations

import math
import os

import numpy as np

from oracle import tdvp_oracle as orc
from oracle import two_site_oracle as tso

TRACE_KINDS = {"H2": 2, "H1b": 3}   # oracle trace labels -> the product's (pytdscf_b200._twosite) trace kinds


def dense_hamiltonian(operators: dict, dims: list[int], coupleJ: complex = 0.0) -> np.ndarray:
    """Sum of the MPO keys as a dense matrix on the product space (site 0 slowest), plus coupleJ times the identity."""
    n = len(dims)
    N = math.prod(dims)
    H = np.eye(N, dtype=complex) * complex(coupleJ)
    for key, cores in operators.items():
        sites = [k[0] if isinstance(k, tuple) else int(k) for k in key]
        by_site = dict(zip(sites, cores, strict=True))
        M = np.ones((1, 1, 1), dtype=complex)        # (bra, ket, w)
        for s in range(n):
            d = dims[s]
            W = by_site.get(s)
            if W is None:
                M = np.einsum("abw,ij->aibjw", M, np.eye(d)).reshape(M.shape[0] * d, M.shape[1] * d, M.shape[2])
                continue
            W = np.asarray(W, dtype=complex)
            if W.ndim == 3:
                F = np.zeros((W.shape[0], d, d, W.shape[2]), dtype=complex)
                F[:, np.arange(d), np.arange(d), :] = W
                W = F
            M = np.einsum("abw,wijt->aibjt", M, W).reshape(M.shape[0] * d, M.shape[1] * d, W.shape[3])
        H += M[:, :, 0]
    return H


def dense_state(cores) -> np.ndarray:
    v = np.asarray(cores[0])[0]
    for c in cores[1:]:
        v = np.tensordot(v, np.asarray(c), axes=(v.ndim - 1, 0))
    return v.reshape(-1)


def random_canonical_mps(dims: list[int], seed: int) -> list[np.ndarray]:
    """Random MPS with full bond dimensions, right-canonical with the centre at site 0 and unit norm."""
    rng = np.random.default_rng(seed)
    n = len(dims)
    big = math.prod(dims)
    cores = []
    for i in range(n):
        ml, mr = orc.bond_dims(dims, i, big)
        shape = (1 if i == 0 else ml, dims[i], 1 if i == n - 1 else mr)
        cores.append(rng.standard_normal(shape) + 1j * rng.standard_normal(shape))
    for i in range(n - 1, 0, -1):
        sig, B = orc.shift_lq(cores[i])
        cores[i] = B
        cores[i - 1] = np.tensordot(cores[i - 1], sig, axes=(2, 0))
    cores[0] = cores[0] / np.linalg.norm(cores[0])
    return cores


def complex_mpo_case() -> dict:
    """A three-site chain (d = 3, 4, 3) whose Hamiltonian is complex Hermitian, not real symmetric: one MPO key, the
    direct sum of a random complex MPO and its adjoint (scaled to spectral norm ~1)."""
    from pytdscf_b200._mps_cuda import direct_sum_mpo

    rng = np.random.default_rng(11)
    dims, w = [3, 4, 3], [1, 2, 2, 1]
    cores = [(rng.standard_normal((w[i], d, d, w[i + 1])) + 1j * rng.standard_normal((w[i], d, d, w[i + 1]))) * 0.3
             for i, d in enumerate(dims)]
    adj = [np.ascontiguousarray(np.conj(W).transpose(0, 2, 1, 3)) for W in cores]
    merged = direct_sum_mpo([cores, adj])
    ops = {((0, 0), (1, 1), (2, 2)): merged}
    H = dense_hamiltonian(ops, dims)
    nrm = np.linalg.norm(H, 2)
    ops = {k: [c / nrm ** (1 / 3) for c in v] for k, v in ops.items()}
    return {"name": "complex3", "dims": dims, "operators": ops, "coupleJ": 0.0}


def oracle_two_site(g: dict, init, *, bond_dim, p_svd, thresh, integrator, conserve_norm=True, space="hilbert"):
    H = orc.MPOHamiltonian(len(g["dims"]), g["operators"], g["coupleJ"])
    return tso.TwoSiteOracle(H, [np.array(c, dtype=complex) for c in init], thresh=thresh, integrator=integrator,
                               conserve_norm=conserve_norm, space=space, bond_dim=bond_dim, p_svd=p_svd)


def oracle_run(g: dict, nstep: int, *, p_svd=1.0e-07, thresh=None, record=True):
    """TwoSiteOracle.propagate_two_site on a golden case from its initial MPS, with the per-step observables the Simulator
    records (state BEFORE each step) and the bond dimensions."""
    o = oracle_two_site(g, g["init"], bond_dim=g["bond_dim"], p_svd=p_svd, thresh=g["thresh_sil"] if thresh is None else thresh,
                        integrator=g["integrator"], conserve_norm=g["conserve_norm"], space=g["space"])
    rows = []
    for _ in range(nstep):
        if record:
            rows.append({"autocorr": o.autocorr(), "energy": o.energy() if g["space"] == "hilbert" else None, "norm": o.norm(),
                         "bonddim": o.bonddim()})
        o.propagate_two_site(g["dt_au"])
    return o, rows


def build_product_model(g: dict):
    """pytdscf_b200 Model of a golden case (as tests/test_gpu_propagation.py::build_model, without gates)."""
    import pytdscf_b200 as tb

    basis = [tb.Exciton(nstate=d) for d in g["dims"]]
    pot = {key: tb.TensorOperator(mpo=[np.asarray(c) for c in cores]) for key, cores in g["operators"].items()}
    if g["coupleJ"] != 0:
        pot[()] = g["coupleJ"]
    ham = tb.TensorHamiltonian(ndof=len(basis), potential=[[pot]], backend="cuda")
    return tb.Model(basis, {"hamiltonian": ham}, bond_dim=g["bond_dim"], space=g["space"])


def product_run(g: dict, tmp_path, nstep: int, *, eng=None, p_svd=1.0e-07, thresh=None, merge=False, **kw):
    """Simulator.propagate(two_site=True) from the golden initial MPS; ``eng`` injects an engine (CPU host-logic tests)."""
    import pytdscf_b200 as tb

    model = build_product_model(g)
    os.chdir(tmp_path)
    sim = tb.Simulator(g["name"] + "_2s", model, backend="cuda")
    if eng is not None:
        sim.eng = eng
    sim.merge_mpo_terms = merge
    sim.set_initial_mps(g["init"])
    hil = g["space"] == "hilbert"
    ener, wf = sim.propagate(stepsize=g["dt_au"] * tb.units.au_in_fs, maxstep=nstep,
                             thresh_sil=g["thresh_sil"] if thresh is None else thresh, integrator=g["integrator"],
                             conserve_norm=g["conserve_norm"], energy=hil, autocorr=True, norm=True, populations=hil,
                             record_trace=True, two_site=True, two_site_p_svd=p_svd, **kw)
    return sim, ener, wf


def recording_split(p_svd: float, margins: list):
    """A wrapper of the oracle's split that records, per call, min_i |cumsum(s)_i / sum(s) - (1 - p)|."""
    inner = tso.split_two_site

    def split(theta, direction, p, Dcap, conserve_norm):
        out = inner(theta, direction, p, Dcap, conserve_norm)
        s = out[2]
        cs = np.cumsum(s)
        if cs[-1] > 0:
            margins.append(float(np.min(np.abs(cs / cs[-1] - (1.0 - p)))))
        return out

    return split
