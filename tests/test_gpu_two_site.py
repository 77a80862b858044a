"""Two-site TDVP on the GPU: tdvp_heff2_apply against einsum, tdvp_krylov_expm2 against the reference Krylov solvers,
tdvp_split2 against LAPACK, and Simulator.propagate(two_site=True) against TwoSiteOracle.propagate_two_site."""
import json
import os

import numpy as np
import pytest
import scipy.linalg

from oracle import tdvp_oracle as orc
from oracle import two_site_oracle as tso
from tests.golden_io import GOLDEN_DIR, RUN_CASES, load_run
from tests.two_site_cases import (TRACE_KINDS, complex_mpo_case, dense_hamiltonian, dense_state, oracle_run, oracle_two_site,
                                  product_run, random_canonical_mps)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from pytdscf_b200._engine import Engine

    e = Engine(0)
    yield e
    e.close()


def crand(rng, *shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / np.sqrt(2)


def _core(rng, kind, wl, d, wr):
    if kind == "id":
        return None
    return crand(rng, wl, d, wr) if kind == "diag" else crand(rng, wl, d, d, wr)


def _run_heff2(eng, terms_np, theta, id_promise=None):
    """terms_np: [(L, W1, W2, R, coef)] host arrays (None = identity) -> device result and einsum reference."""
    dev_terms, ref_terms = [], []
    for L, W1, W2, R, coef in terms_np:
        c1, c2 = eng.upload_core(W1), eng.upload_core(W2)
        if id_promise is not None:
            c1.l_id, c2.r_id = id_promise
        dev_terms.append((None if L is None else eng.to_device(L), c1, c2, None if R is None else eng.to_device(R), coef))
        ref_terms.append((L, None if W1 is None else orc.SiteCore((), 0, W1, False, False),
                          None if W2 is None else orc.SiteCore((), 0, W2, False, False), R, coef))
    out = eng.heff2_apply(dev_terms, eng.to_device(theta)).cpu().numpy()
    return out, tso.heff2_apply(ref_terms, theta)


def _rel(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


@pytest.mark.parametrize("k1", ["id", "diag", "full"])
@pytest.mark.parametrize("k2", ["id", "diag", "full"])
def test_heff2_core_kinds(eng, k1, k2):
    kinds = ["id", "diag", "full"]
    rng = np.random.default_rng(3 * kinds.index(k1) + kinds.index(k2))
    Dl, d1, d2, Dr = 7, 3, 5, 6
    wl = 1 if k1 == "id" else 3
    wr = 1 if k2 == "id" else 4
    wm = 1 if (k1 == "id" or k2 == "id") else 2
    theta = crand(rng, Dl, d1, d2, Dr)
    terms = [(crand(rng, Dl, wl, Dl), _core(rng, k1, wl, d1, wm), _core(rng, k2, wm, d2, wr), crand(rng, Dr, wr, Dr), 0.7 - 0.3j),
             (None, None, None, crand(rng, Dr, 1, Dr), 1.0)]
    out, ref = _run_heff2(eng, terms, theta)
    assert _rel(out, ref) <= 1e-12


@pytest.mark.parametrize("shape", [(1, 2, 3, 1), (5, 4, 2, 9), (1, 3, 3, 8), (256, 4, 4, 256)])
def test_heff2_blocks_and_shapes(eng, shape):
    """L / R absent or present, D = 1, D_l != D_r, d1 != d2, and a TMA-eligible D = 256, d = 4 pair."""
    rng = np.random.default_rng(sum(shape))
    Dl, d1, d2, Dr = shape
    theta = crand(rng, *shape)
    w = 3
    terms = [(None, crand(rng, 1, d1, d1, w), crand(rng, w, d2, d2, 1), None, 1.0),
             (crand(rng, Dl, w, Dl), crand(rng, w, d1, 2), crand(rng, 2, d2, d2, 1), None, 2.0j),
             (None, crand(rng, 1, d1, 2), crand(rng, 2, d2, d2, w), crand(rng, Dr, w, Dr), 1.0),
             (crand(rng, Dl, 1, Dl), None, None, crand(rng, Dr, 1, Dr), -0.5),
             (None, None, None, None, 0.25)]
    out, ref = _run_heff2(eng, terms, theta)
    assert _rel(out, ref) <= 1e-12


@pytest.mark.parametrize("promise", [False, True])
def test_heff2_identity_channels(eng, promise):
    """theta above 2^17 elements; with the promise the named channels of L and R are unit matrices and are copied."""
    rng = np.random.default_rng(3)
    Dl, d1, d2, Dr, w = 64, 6, 6, 64, 4
    theta = crand(rng, Dl, d1, d2, Dr)
    assert theta.size >= 2**17
    L, R = crand(rng, Dl, w, Dl), crand(rng, Dr, w, Dr)
    L[:, 0, :] = np.eye(Dl)
    R[:, w - 1, :] = np.eye(Dr)
    terms = [(L, crand(rng, w, d1, d1, 2), crand(rng, 2, d2, w), R, 1.0 + 0.5j)]
    out, ref = _run_heff2(eng, terms, theta, id_promise=(0, w - 1) if promise else None)
    assert _rel(out, ref) <= 1e-12


def test_heff2_equals_one_site_on_the_merged_index_and_profiles_its_stages(eng):
    rng = np.random.default_rng(9)
    Dl, d1, d2, Dr, wl, wm, wr = 24, 3, 4, 20, 3, 2, 5
    theta = crand(rng, Dl, d1, d2, Dr)
    L, R = crand(rng, Dl, wl, Dl), crand(rng, Dr, wr, Dr)
    W1, W2 = crand(rng, wl, d1, d1, wm), crand(rng, wm, d2, d2, wr)
    Wm = np.einsum("cijt,tklu->cikjlu", W1, W2).reshape(wl, d1 * d2, d1 * d2, wr)
    eng.gemm_profile(True, reset=True)
    two = eng.heff2_apply([(eng.to_device(L), eng.upload_core(W1), eng.upload_core(W2), eng.to_device(R), 1.0)],
                          eng.to_device(theta)).cpu().numpy()
    eng.gemm_profile(False)
    labels = eng.profile_breakdown()
    one = eng.heff_apply([(eng.to_device(L), eng.upload_core(Wm), eng.to_device(R), 1.0)],
                         eng.to_device(theta.reshape(Dl, d1 * d2, Dr))).cpu().numpy()
    assert _rel(two.reshape(one.shape), one) <= 1e-12
    text = json.dumps(labels)
    for s in ("heff2.s1", "heff2.s2", "heff2.s3", "heff2.s4"):
        assert s in text, labels


@pytest.mark.parametrize("hermitian", [True, False])
@pytest.mark.parametrize("shape", [(16, 8, 8, 16), (32, 8, 8, 32)])
def test_krylov_expm2_matches_reference_solvers(eng, hermitian, shape):
    """N = 16 384 and 65 536: both sides of the fused small-vector Lanczos switch (32 768)."""
    rng = np.random.default_rng(shape[0] + hermitian)
    Dl, d1, d2, Dr = shape
    w = 2
    L = crand(rng, Dl, 1, Dl)
    R = crand(rng, Dr, 1, Dr)
    W1 = crand(rng, 1, d1, d1, w)
    W2 = crand(rng, w, d2, d2, 1)
    if hermitian:
        L = 0.5 * (L + np.conj(L.transpose(2, 1, 0)))
        R = 0.5 * (R + np.conj(R.transpose(2, 1, 0)))
        W1 = 0.5 * (W1 + np.conj(W1.transpose(0, 2, 1, 3)))
        W2 = 0.5 * (W2 + np.conj(W2.transpose(0, 2, 1, 3)))
    terms_np = [(None, W1, W2, None, 1.0), (L, None, None, R, 1.0)]
    ref_terms = [(a, None if b is None else orc.SiteCore((), 0, b, False, False),
                  None if c is None else orc.SiteCore((), 0, c, False, False), d, e) for a, b, c, d, e in terms_np]
    theta = crand(rng, *shape)
    theta /= np.linalg.norm(theta)
    x = theta
    for _ in range(30):        # power iteration: |H2| to a few per cent, so that |scale H2| stays near 1/2
        y = tso.heff2_apply(ref_terms, x)
        nrm = float(np.linalg.norm(y))
        x = y / nrm
    dev_terms = [(None if a is None else eng.to_device(a), eng.upload_core(b), eng.upload_core(c),
                  None if d is None else eng.to_device(d), e) for a, b, c, d, e in terms_np]
    for kind, solver in (("lanczos", orc.sil_reference), ("arnoldi", orc.sia_reference)):
        if kind == "lanczos" and not hermitian:
            continue
        for cn in (True, False):
            scale = -0.5j / nrm
            ref, n_ref = solver(scale, lambda x: tso.heff2_apply(ref_terms, x), theta, 1e-10, conserve_norm=cn)
            t = eng.to_device(theta)
            n = eng.krylov_expm2(kind, scale, 1e-10, 0, cn, t, dev_terms)
            assert n == n_ref
            assert np.abs(t.cpu().numpy() - ref).max() <= 1e-11


@pytest.mark.parametrize("shape,rank_def,p,cap", [
    ((4, 5, 3, 2), False, 0.0, 100), ((3, 2, 6, 7), False, 1e-3, 100), ((6, 4, 3, 8), False, 0.0, 5),
    ((5, 6, 6, 5), True, 0.0, 100), ((2, 3, 8, 9), True, 1e-6, 100), ((16, 16, 16, 16), False, 0.05, 40)])
@pytest.mark.parametrize("direction", ["left", "right"])
def test_split2_matches_lapack(eng, shape, rank_def, p, cap, direction):
    rng = np.random.default_rng(sum(shape))
    Dl, d1, d2, Dr = shape
    m, n = Dl * d1, d2 * Dr
    M = crand(rng, m, n)
    if rank_def:
        M = crand(rng, m, 3) @ crand(rng, 3, n)      # rank 3: the other singular values vanish
        M[:, 0] = 0.0
    theta = M.reshape(shape)
    U, s, Vh = np.linalg.svd(M, full_matrices=False)
    for cn in (True, False):
        left, right, s_dev, r = eng.split2(direction, eng.to_device(theta), p, cap, cn)
        left, right = left.cpu().numpy(), right.cpu().numpy()
        _l, _r, _s, r_ref = tso.split_two_site(theta, direction, p, cap, cn)
        if rank_def and p == 0.0:
            # exact zeros: which rounding-level values still move the cumulative sum is unpinned on either side;
            # they carry nothing, so the reconstruction below must agree regardless
            assert r >= 3 and r_ref >= 3
        else:
            assert r == r_ref
        big = s > 1e-8 * s[0]
        assert np.abs(s_dev[big] - s[big]).max() <= 1e-12 * s[0]
        rec = np.tensordot(left, right, axes=(2, 0))
        rec_ref = np.tensordot(_l, _r, axes=(2, 0))
        assert np.abs(rec - rec_ref).max() <= 1e-12 * s[0]
        iso = left.reshape(m, r) if direction == "right" else right.reshape(r, n).conj().T
        assert np.abs(iso.conj().T @ iso - np.eye(r)).max() <= 1e-13


def _noise_floor(name):
    nf = json.load(open(os.path.join(GOLDEN_DIR, "noise_floor_two_site.json")))[name]
    return {"autocorr": max(1e-10, 4 * nf["autocorr_abs"]), "energy": max(1e-10, 4 * nf["energy_rel"]),
            "state": max(1e-10, 4 * nf["state_abs"])}


NSTEP = 5


@pytest.mark.parametrize("name", RUN_CASES)
def test_two_site_propagation_matches_oracle(name, tmp_path):
    g = load_run(name)
    o, rows = oracle_run(g, NSTEP)
    sim, ener, wf = product_run(g, tmp_path, NSTEP)
    tol = _noise_floor(name)
    assert [tuple(t) for t in wf.ci_coef.trace] == [(TRACE_KINDS[k], s, n) for k, s, n in o.trace]
    for rec, row in zip(sim.history, rows, strict=True):
        assert rec["bonddim"] == row["bonddim"]
        assert abs(rec["autocorr"] - row["autocorr"]) <= tol["autocorr"] * max(1.0, abs(row["autocorr"]))
        assert abs(rec["norm"] - row["norm"]) <= max(1e-10, tol["state"])
        if g["space"] == "hilbert":
            assert abs(rec["energy"] - row["energy"]) <= tol["energy"] * abs(row["energy"])
    lines = open(os.path.join(g["name"] + "_2s_prop", "bonddim.dat")).read().splitlines()
    assert [[int(b) for b in ln.split()[1:]] for ln in lines[1:]] == [r["bonddim"] for r in rows]
    a, b = dense_state(wf.ci_coef.to_numpy()), dense_state(o.mps)
    assert np.abs(a - b).max() <= tol["state"] * max(1.0, np.abs(b).max())


@pytest.mark.parametrize("name", ["henon_heiles_f2", "exciton_D2", "complex3"])
def test_two_site_is_exact_on_the_device(name, tmp_path):
    """Full bond dimension, p = 0, Arnoldi at 1e-14: 10 steps on the GPU equal expm(-iHt) psi0 to 1e-9."""
    import pytdscf_b200 as tb

    g = complex_mpo_case() if name == "complex3" else load_run(name)
    H = dense_hamiltonian(g["operators"], g["dims"], g["coupleJ"])
    init = random_canonical_mps(g["dims"], 3)
    dt = 1.0 / np.linalg.norm(H, 2)
    basis = [tb.Exciton(nstate=d) for d in g["dims"]]
    pot = {k: tb.TensorOperator(mpo=[np.asarray(c) for c in v]) for k, v in g["operators"].items()}
    if g["coupleJ"] != 0:
        pot[()] = g["coupleJ"]
    model = tb.Model(basis, {"hamiltonian": tb.TensorHamiltonian(ndof=len(basis), potential=[[pot]], backend="cuda")},
                     bond_dim=int(np.prod(g["dims"])))
    os.chdir(tmp_path)
    sim = tb.Simulator("exact", model)
    sim.set_initial_mps(init)
    _, wf = sim.propagate(stepsize=dt * tb.units.au_in_fs, maxstep=10, thresh_sil=1e-14, integrator="arnoldi",
                          two_site=True, two_site_p_svd=0.0, write_files=False)
    ref = scipy.linalg.expm(-1j * H * 10 * dt) @ dense_state(init)
    assert np.abs(dense_state(wf.ci_coef.to_numpy()) - ref).max() <= 1e-9


def test_two_site_restart_continues_the_run(tmp_path):
    """5 steps, save, restart, 5 more = 10 steps in one go, to 1e-12 (thresh 1e-14: the restarted run's empty warm-up
    history then changes nothing above rounding)."""
    g = load_run("henon_heiles_f6")
    _, _, wf10 = product_run(g, tmp_path, 10, thresh=1e-14, write_files=False)
    sim, _, wf5 = product_run(g, tmp_path, 5, thresh=1e-14, savefile_ext="_half")
    import pytdscf_b200 as tb

    sim2 = tb.Simulator(g["name"] + "_2s", sim.model)
    _, wf = sim2.propagate(stepsize=g["dt_au"] * tb.units.au_in_fs, maxstep=5, restart=True, loadfile_ext="_half",
                           thresh_sil=1e-14, two_site=True, write_files=False)
    assert wf.ci_coef.bonddim() == wf10.ci_coef.bonddim()
    a, b = dense_state(wf.ci_coef.to_numpy()), dense_state(wf10.ci_coef.to_numpy())
    assert np.abs(a - b).max() <= 1e-12


def test_krylov_expm2_reports_an_oversize_basis(eng):
    """A theta whose Krylov basis exceeds the device memory returns TDVP_ERR_NO_MEMORY with the size, not a CUDA error."""
    import ctypes as C

    from pytdscf_b200 import _lib

    theta = eng.empty(1, 1, 1, 1)
    arr = eng.heff2_terms([(None, None, None, None, 1.0)])
    niter = C.c_int(0)
    Dl = Dr = 8192
    d = 64     # the vector alone: 8192^2 * 64^2 * 16 B = 4.4 TB; theta's pointer is never read
    rc = eng.lib.tdvp_krylov_expm2(eng.h, 0, 0.0, -0.1, 1e-9, 0, 1, arr, 1, Dl, d, d, Dr, C.c_void_p(theta.data_ptr()),
                                   C.byref(niter))
    assert rc == _lib.ERR_NO_MEMORY
    assert "GB" in eng.lib.tdvp_last_error(eng.h).decode()
    # the handle still works
    t = eng.to_device(np.ones((2, 2, 2, 2), dtype=complex) / 4)
    assert eng.krylov_expm2("lanczos", -0.1j, 1e-9, 0, True, t, [(None, None, None, None, 1.0)]) >= 1
