"""GPU parity tests, propagation level: Simulator(backend="cuda") against golden runs of the UNMODIFIED
reference (tests/golden/*.npz) -- identical Krylov traces, per-step energy / autocorrelation / norm within
1e-10 relative (the north-star tolerance for complex128), final MPS tensors, and the oracle re-run on the box."""
import os

import numpy as np
import pytest

from oracle import tdvp_oracle as orc
from tests.golden_io import GATE_CASES, RUN_CASES, load_run

pytestmark = pytest.mark.gpu
REL = 1e-10  # north-star tolerance (complex128)


def tolerances(name):
    """max(1e-10, 4 x the reference algorithm's own rounding-noise floor) per observable.

    tests/golden/noise_floor.json (made by tests/golden/make_noise_floor.py) records how far the reference
    algorithm moves when its H_eff outputs are perturbed by one rounding (2e-16 relative): for well-conditioned
    cases that is ~1e-15 and the bar is the plain 1e-10; exciton_D6 (bond dimension 6 on a state of numerical
    rank ~2) is ill-conditioned -- 1e-8 in the autocorrelation -- and no implementation, the reference with
    another BLAS included, can agree better than that (SURVEY F7)."""
    import json

    from tests.golden_io import GOLDEN_DIR

    nf = json.load(open(os.path.join(GOLDEN_DIR, "noise_floor.json")))[name]
    return {"autocorr": max(REL, 4 * nf["autocorr_abs"]), "energy": max(REL, 4 * nf["energy_rel"]),
            "state": max(1e-9, 4 * nf["state_abs"])}


def dense_state(cores):
    """Contract an MPS to the full coefficient vector (gauge invariant; small systems only)."""
    v = np.asarray(cores[0])[0]  # (d, Dr)
    for c in cores[1:]:
        v = np.tensordot(v, np.asarray(c), axes=(v.ndim - 1, 0))
    return v.reshape(-1)


def assert_same_state(cores, ref_cores, tol=1e-9):
    """Site tensors themselves are gauge-conditioned (a bond direction of weight s carries rounding ~1e-16/s),
    so parity of the final wavefunction is asserted on the contracted state vector."""
    for c, r in zip(cores, ref_cores, strict=True):
        assert np.asarray(c).shape == np.asarray(r).shape  # identical (static) bond dimensions
    a, b = dense_state(cores), dense_state(ref_cores)
    assert np.abs(a - b).max() <= tol * max(1.0, np.abs(b).max())


def build_model(g):
    import pytdscf_b200 as tb

    basis = [tb.Exciton(nstate=d) for d in g["dims"]]
    pot = {}
    for key, cores in g["operators"].items():
        pot[key] = tb.TensorOperator(mpo=[np.asarray(c) for c in cores])
    if g["coupleJ"] != 0:
        pot[()] = g["coupleJ"]
    ham = tb.TensorHamiltonian(ndof=len(basis), potential=[[pot]], backend="cuda")
    gate = None
    if g.get("gates"):
        gp = {}
        for site, U in g["gates"].items():
            if U.ndim == 1:
                gp[(site,)] = tb.TensorOperator(mpo=[U.reshape(1, -1, 1)], legs=(site,))
            else:
                gp[((site, site),)] = tb.TensorOperator(mpo=[U.reshape(1, U.shape[0], U.shape[1], 1)], legs=(site, site))
        gate = tb.TensorHamiltonian(ndof=len(basis), potential=[[gp]], backend="cuda")
    return tb.Model(basis, {"hamiltonian": ham}, bond_dim=g["bond_dim"], space=g["space"], one_gate_to_apply=gate)


def run_cuda(g, tmp_path, use_golden_init=True):
    import pytdscf_b200 as tb

    model = build_model(g)
    if g["hartree"] is not None and not use_golden_init:
        model.init_HartreeProduct = [[h for h in g["hartree"]]]
    os.chdir(tmp_path)
    sim = tb.Simulator(g["name"], model, backend="cuda", verbose=2)
    if use_golden_init:
        sim.set_initial_mps(g["init"])
    hil = g["space"] == "hilbert"
    ener, wf = sim.propagate(stepsize=g["dt_au"] * tb.units.au_in_fs, maxstep=g["nstep"], thresh_sil=g["thresh_sil"],
                             integrator=g["integrator"], conserve_norm=g["conserve_norm"], energy=hil, autocorr=hil,
                             norm=hil, populations=hil, record_trace=True)
    return sim, ener, wf


@pytest.mark.parametrize("name", RUN_CASES + GATE_CASES)
def test_propagation_matches_reference(name, tmp_path):
    g = load_run(name)
    sim, ener, wf = run_cuda(g, tmp_path)
    trace = np.array(wf.ci_coef.trace)
    assert trace.shape == g["trace"].shape and (trace == g["trace"]).all(), "Krylov iteration trace differs"
    tol = tolerances(name)
    if g["space"] == "hilbert":
        for rec, row in zip(sim.history, g["props"], strict=True):
            t, ar, ai, er, ei, nrm = row
            assert abs(rec["autocorr"] - complex(ar, ai)) <= tol["autocorr"] * max(1.0, abs(complex(ar, ai)))
            assert abs(rec["energy"] - er) <= tol["energy"] * abs(er)
            assert abs(rec["norm"] - nrm) <= REL
            assert abs(rec["pops"][0] - nrm**2) <= REL
        assert abs(ener - g["final_energy"].real) <= tol["energy"] * abs(g["final_energy"].real)
    assert_same_state(wf.ci_coef.to_numpy(), g["final"], tol["state"])
    # output files in the reference layout
    assert os.path.exists(os.path.join(g["name"] + "_prop", "main.log"))
    if g["space"] == "hilbert":
        lines = open(os.path.join(g["name"] + "_prop", "autocorr.dat")).read().splitlines()
        assert lines[0].startswith("# time [fs]") and len(lines) == g["nstep"] + 1


@pytest.mark.parametrize("name", ["exciton_D2", "exciton_D6", "liouville_spin3"])
def test_device_initial_mps_matches_reference(name, tmp_path):
    """alloc_random on the device (LQ sweeps through tdvp_qr_shift) reproduces the reference's initial MPS,
    including LAPACK's null-space completion of the zero-padded Hartree product."""
    from pytdscf_b200._engine import Engine
    from pytdscf_b200._mps_cuda import MPSCoefCuda

    g = load_run(name)
    model = build_model(g)
    model.init_HartreeProduct = [[h for h in g["hartree"]]]
    eng = Engine(0)
    mps = MPSCoefCuda.alloc_random(eng, model)
    for c, r in zip(mps.to_numpy(), g["init"], strict=True):
        assert c.shape == r.shape
        np.testing.assert_allclose(c, r, rtol=0, atol=1e-13)
    eng.close()


def test_full_api_with_ho_dvr_basis(tmp_path):
    """End-to-end through the public API with HO-DVR primitives (default initial state, FBR->DVR unitary)
    on the H2CO golden case (BASELINE config 1): the initial MPS and the propagation match the reference."""
    import pytdscf_b200 as tb

    g = load_run("h2co_D16")
    freqs = [1186.325, 1252.832, 1514.908, 1831.831, 2863.96, 2916.722]
    prims = [tb.HarmonicOscillator(5, f, units="cm-1") for f in freqs]
    keys = list(g["operators"])
    pot_cores, kin_cores = g["operators"][keys[0]], g["operators"][keys[1]]
    model = tb.Model(prims, {"potential": pot_cores, "kinetic": kin_cores}, bond_dim=16)
    os.chdir(tmp_path)
    sim = tb.Simulator("h2co_api", model, backend="cuda")
    ener, wf = sim.propagate(stepsize=0.1, maxstep=g["nstep"], record_trace=True)
    assert (np.array(wf.ci_coef.trace) == g["trace"]).all()
    assert abs(ener - g["final_energy"].real) <= REL * abs(g["final_energy"].real)
    for rec, row in zip(sim.history, g["props"], strict=True):
        assert abs(rec["autocorr"] - complex(row[1], row[2])) <= REL


def test_oracle_rerun_on_this_box_agrees(tmp_path):
    """SURVEY F7: assert against the oracle run on the same box, not only against stored literals."""
    g = load_run("henon_heiles_f6")
    H = orc.MPOHamiltonian(len(g["dims"]), g["operators"], g["coupleJ"])
    o = orc.TDVPOracle(H, [c.copy() for c in g["init"]], thresh=g["thresh_sil"])
    e_or = []
    for _ in range(g["nstep"]):
        e_or.append(o.expectation().real)
        o.propagate(g["dt_au"])
    sim, ener, wf = run_cuda(g, tmp_path)
    for rec, e in zip(sim.history, e_or, strict=True):
        assert abs(rec["energy"] - e) <= REL * abs(e)
    assert_same_state(wf.ci_coef.to_numpy(), o.mps)


def test_backend_switch_errors():
    import pytdscf_b200 as tb

    g = load_run("exciton_D2")
    model = build_model(g)
    with pytest.raises(ValueError):
        tb.Simulator("x", model, backend="numpy")
    with pytest.raises(ValueError):
        tb.TensorHamiltonian(ndof=1, potential=[[{}]], backend="tensorflow")


def run_relax(g, tmp_path, improved):
    import pytdscf_b200 as tb

    model = build_model(g)
    os.chdir(tmp_path)
    sim = tb.Simulator(g["name"], model, backend="cuda")
    sim.set_initial_mps(g["init"])
    ener, wf = sim.relax(stepsize=g["dt_au"] * tb.units.au_in_fs, maxstep=g["nstep"], improved=improved, record_trace=True)
    return sim, ener, wf


def test_imaginary_time_relaxation_matches_reference(tmp_path):
    g = load_run("relax_imag_hh4")
    sim, ener, wf = run_relax(g, tmp_path, improved=False)
    assert (np.array(wf.ci_coef.trace) == g["trace"]).all()
    for rec, row in zip(sim.history, g["props"], strict=True):
        assert abs(rec["energy"] - row[3]) <= REL * abs(row[3])
        assert abs(rec["norm"] - row[5]) <= REL
    assert_same_state(wf.ci_coef.to_numpy(), g["final"])


def test_improved_relaxation_matches_reference(tmp_path):
    """Per-site Lanczos eigen-solves.  The reference takes the Ritz vector from scipy's eigh_tridiagonal whose SIGN is
    LAPACK-internal (unpinned); we fix a positive overlap with the previous vector, so Lanczos dimensions may differ by
    one where LAPACK flips a sign, and agreement is at the solver's convergence threshold (1e-9), phase excluded."""
    g = load_run("relax_improved_hh4")
    sim, ener, wf = run_relax(g, tmp_path, improved=True)
    tr = np.array(wf.ci_coef.trace)
    assert tr.shape == g["trace"].shape and (tr[:, :2] == g["trace"][:, :2]).all()  # same sequence of solves (no K solves)
    # where LAPACK's arbitrary eigenvector sign flips between two Lanczos iterations the reference sees |dy| ~ 2 and
    # keeps iterating (typically 4 vectors on an already converged site where 2 suffice); never the other way round
    big = g["trace"][:, 2] > 4
    assert (tr[:, 2] <= g["trace"][:, 2] + 1).all()
    assert np.abs(tr[big, 2] - g["trace"][big, 2]).max() <= 1
    for rec, row in zip(sim.history, g["props"], strict=True):
        assert abs(rec["energy"] - row[3]) <= 1e-9 * abs(row[3])
        assert abs(rec["norm"] - row[5]) <= REL
    assert abs(ener - g["final_energy"].real) <= 1e-9 * abs(g["final_energy"].real)
    a, b = dense_state(wf.ci_coef.to_numpy()), dense_state(g["final"])
    assert abs(abs(np.vdot(a, b)) - 1.0) <= 1e-9


def test_reduced_densities_gpu():
    """Device reduced densities (two DMMA GEMMs per site) against the reference's get_reduced_densities goldens."""
    from pytdscf_b200._engine import Engine
    from pytdscf_b200._mps_cuda import MPSCoefCuda

    eng = Engine(0)
    from tests.golden_io import load_run
    from tests.rdm_cases import check_rdms

    check_rdms(eng, load_run, MPSCoefCuda, atol=1e-13)


@pytest.mark.parametrize("case", ["kraus_spin4", "kraus2_spin4"])
def test_kraus_map_gpu(case, tmp_path):
    """One-site Kraus map on a purified MPS (device GEMM + Jacobi SVD) against the reference run: Krylov trace, per-step
    energy / norm and the system reduced density of the Kraus site (ancilla phases are an SVD gauge, traced out)."""
    import pytdscf_b200 as tb
    from tests.test_host_sweep_cpu import _kraus_model, kraus_observables

    g = load_run(case)
    os.chdir(tmp_path)
    sim = tb.Simulator("kraus_gpu", _kraus_model(g), backend="cuda")
    sim.set_initial_mps(g["init"])
    ener, wf = sim.propagate(stepsize=g["dt_au"] * tb.units.au_in_fs, maxstep=g["nstep"], autocorr=False, populations=False,
                             conserve_norm=False, record_trace=True)
    assert (np.array(wf.ci_coef.trace) == g["trace"]).all()
    obs, rho, ref = kraus_observables(sim, wf, g)
    for (e, n), row in zip(obs, g["props"], strict=True):
        assert abs(e - row[3]) <= REL * max(1.0, abs(row[3])) and abs(n - row[5]) <= REL
    np.testing.assert_allclose(rho, ref, atol=1e-10)


@pytest.mark.parametrize("case", ["adaptive_exciton", "adaptive_hh6"])
def test_adaptive_tdvp_gpu(case, tmp_path):
    """Rank-adaptive one-site TDVP on the device (square kernels on zero-padded operands, Householder completion for the
    new bond directions, Krylov size override): same bond growth, Krylov trace and observables as the reference."""
    from tests.test_host_sweep_cpu import run_adaptive

    g = load_run(case)
    sim, ener, wf = run_adaptive(g, None, tmp_path, "_gpu")
    assert [s.shape for s in wf.ci_coef.sites] == [c.shape for c in g["final"]]
    assert (np.array(wf.ci_coef.trace) == g["trace"]).all()
    tol = tolerances(g["name"])
    for rec, row in zip(sim.history, g["props"], strict=True):
        assert abs(rec["autocorr"] - complex(row[1], row[2])) <= tol["autocorr"]
        assert abs(rec["energy"] - row[3]) <= tol["energy"] * abs(row[3]) and abs(rec["norm"] - row[5]) <= REL
    assert_same_state(wf.ci_coef.to_numpy(), g["final"], tol["state"])


@pytest.mark.parametrize("tag", ["full", "sub"])
def test_liouville_observables_and_subspace(tag, tmp_path):
    """Liouville space on the GPU: Tr(O rho) of three Hilbert-space observables per step (reference ``_exp_liouville``,
    pytdscf/_mps_cls.py:3769-3838), norm / populations, and the sub-space projection of the initial MPDO
    (``project_subspace``, pytdscf/_mps_mpo.py:196-220), against goldens of the unmodified reference."""
    from tests.liouville_obs_cases import check_case, run_case

    sim, wf = run_case(tag, tmp_path)
    check_case(tag, sim, wf, tol_expect=REL, tol_state=1e-9)


@pytest.mark.parametrize("tag", ["prop", "rand"])
def test_hermitise_mpdo_gpu(tag):
    """rho <- (rho + rho^dagger) / 2 with re-compression to the original bonds (reference ``MPSCoef.hermitise`` /
    ``svd_conj_mpdo``, _mps_cls.py:2289-2312, 2516-2562) on the device (GEMM + Jacobi SVD per bond, QR re-canonicalisation):
    the dense density operator equals the unmodified reference's (tests/golden/hermitise.npz) to 1e-11 relative."""
    from pytdscf_b200._engine import Engine
    from tests.hermitise_cases import run_and_check

    eng = Engine(0)
    try:
        err, asym = run_and_check(tag, eng, tol=1e-11)
        if tag == "prop":
            assert asym < 1e-11
    finally:
        eng.close()


def test_restart_from_reference_checkpoint_on_gpu(tmp_path):
    """A ``wf_*.pkl`` in the reference's format (its WFunc layout) restarts on the GPU and continues with the reference's
    own energies (tests/golden/make_golden_checkpoint.py), SURVEY 8(f4).  The file holds the reference's state after 3
    steps (``tests.golden_io.write_checkpoint``), from which the reference itself continued exactly as from its own dump."""
    import pytdscf_b200 as tb
    from tests.golden_io import load_checkpoint, write_checkpoint

    g = load_run("exciton_D6")
    os.chdir(tmp_path)
    write_checkpoint("wf_ck.pkl")
    sim = tb.Simulator("ck", build_model(g), backend="cuda", verbose=0)
    ener, wf = sim.propagate(stepsize=0.1, maxstep=3, restart=True, loadfile_ext="", savefile_ext="_cont", autocorr=False,
                             norm=False, populations=False)
    ref = load_checkpoint()["energies_restart_reference_file"]
    for rec, e in zip(sim.history, ref, strict=True):
        assert abs(rec["energy"] - e) <= REL * abs(e)
