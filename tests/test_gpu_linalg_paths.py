"""GPU tests of the QR, SVD, pseudo-inverse and Lanczos kernels on both sides of every size switch between two
implementations, each compared with a plain high-precision reference of the same operation.  Every boundary case also
checks, through the per-label launch profile, that the kernel it targets is the one that ran.

Switches (constants from csrc/qr.cu, csrc/svd.cu, csrc/krylov.cu):
  QR panel       k_qr_panel_cluster while the panel has <= qr_max_cluster x CL_ROWS = 16 x 256 rows, k_qr_panel above,
                 with its slabs in global memory above num_sms x SLAB_ROWS = num_sms x 256 rows
  Jacobi SVD     k_jacobi_svd_blocked when n <= 2B and 2 B m x 16 bytes <= 160 KiB for a block width B in {16, 8, 4, 2},
                 k_jacobi_svd otherwise
  pinv           inputs the device probe finds diagonal are inverted directly, all others go through the SVD
  Lanczos step   the fused cluster kernel k_lanczos_step_small for N <= 32768, three kernels above

Tolerances are multiples of EPS = 2.2e-16 times a dimension factor; each one says where it comes from.
"""
import contextlib

import numpy as np
import pytest

from oracle import tdvp_oracle as orc

pytestmark = pytest.mark.gpu

EPS = 2.220446049250313e-16
CL_ROWS = 256             # rows per CTA of both QR panel kernels (SLAB_ROWS = CL_ROWS)
MAX_CLUSTER = 16          # largest cluster of k_qr_panel_cluster
SVD_SMEM = 160 * 1024     # BJ_SMEM_COLS_BYTES
FUSED_MAX_N = 32768       # FUSED_CLUSTER x FUSED_THREADS x FUSED_PER_THREAD


@pytest.fixture(scope="module")
def eng():
    from pytdscf_b200._engine import Engine

    e = Engine(0)
    yield e
    e.close()


@pytest.fixture(scope="module")
def num_sms():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


@contextlib.contextmanager
def launched(eng):
    """Collects the profile labels of the launches inside the block (recording is process-global: always switched off)."""
    labels = set()
    eng.gemm_profile(True, reset=True)
    try:
        yield labels
        labels.update(eng.profile_breakdown())
    finally:
        eng.gemm_profile(False)


def crand(rng, *shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / np.sqrt(2)


def relerr(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def hermitian(rng, n):
    X = crand(rng, n, n)
    return (X + X.conj().T) / (2 * np.sqrt(n))   # spectral radius ~ 1


def orth(M):
    """max |M^H M - I|"""
    return np.abs(M.conj().T @ M - np.eye(M.shape[1])).max()


# ---------------------------------------------------------------------------------------------------------------------
# 1. SVD of tall rank-deficient matrices: the completion QR runs on all m rows, beyond num_sms x 256 of them
@pytest.mark.parametrize("m,n", [(262144, 8), (65536, 10)])     # regularize_site's (D_l D_r) x d at D = 512 / 256
@pytest.mark.parametrize("nzero", [1, 3])
def test_svd_tall_rank_deficient(eng, num_sms, m, n, nzero):
    assert m > num_sms * CL_ROWS
    rng = np.random.default_rng(m + n + nzero)
    M = crand(rng, m, n)
    M[:, n - nzero:] = 0.0
    with launched(eng) as labels:
        U, s, Vh = eng.svd(eng.to_device(M))
    assert {"svd.k_jacobi_svd", "qr.k_qr_panel"} <= labels
    U, Vh = U.cpu().numpy(), Vh.cpu().numpy()
    s_ref = np.linalg.svd(M, compute_uv=False)
    r = n - nzero
    # Householder / Jacobi orthogonality: a few EPS per column pair, times sqrt(m) for the m-term inner products
    assert orth(U) < 20 * np.sqrt(m) * EPS
    assert orth(Vh.conj().T) < 20 * n * EPS
    # reconstruction: backward error of order sqrt(m) EPS relative to s_max
    assert np.abs((U * s[None, :]) @ Vh - M).max() < 20 * np.sqrt(m) * EPS * s_ref[0]
    np.testing.assert_allclose(s[:r], s_ref[:r], rtol=1e-12)      # Jacobi: relative accuracy, ~ n sqrt(m) EPS
    assert np.all(s[r:] == 0.0)                                    # exactly-zero columns are frozen, never rotated


def test_qr_shift_regularized_tall_site(eng):
    """The site-parallel boundary: qr_shift(regularize=True) of a (512, 8, 512) site whose level 7 is empty."""
    Dl, d, Dr = 512, 8, 512
    rng = np.random.default_rng(7)
    psi = crand(rng, Dl, d, Dr)
    psi[:, 7, :] = 0.0
    A, sig = eng.qr_shift("A", eng.to_device(psi), regularize=True)
    A, sig = A.cpu().numpy(), sig.cpu().numpy()
    assert orth(A.reshape(Dl * d, Dr)) < 20 * np.sqrt(Dl * d) * EPS
    Mreg = np.tensordot(A, sig, axes=(2, 0)).transpose(0, 2, 1).reshape(Dl * Dr, d)   # A.sigma = psi_reg, matricised
    U, s, Vh = np.linalg.svd(psi.transpose(0, 2, 1).reshape(Dl * Dr, d), full_matrices=False)
    r = d - 1
    s_reg = np.where(s > 1e-4, s, s + 1e-4 * np.exp(-s / 1e-4))
    # the input's singular vectors span psi_reg's range with the floored values; the completion vector is gauge-free,
    # so only projections are compared.  Scale: ~ sqrt(Dl Dr) EPS relative to s_max (two GEMMs, one QR)
    tol = 100 * np.sqrt(Dl * Dr) * EPS * s[0]
    assert np.abs(U[:, :r].conj().T @ Mreg - s_reg[:r, None] * Vh[:r]).max() < tol
    assert np.abs(Mreg @ Vh[:r].conj().T - U[:, :r] * s_reg[None, :r]).max() < tol
    assert np.abs(np.linalg.svd(Mreg, compute_uv=False) - s_reg).max() < tol


# ---------------------------------------------------------------------------------------------------------------------
# 2. QR: which panel kernel runs at the switch, and one factorisation that uses both
@pytest.mark.parametrize("rows,kernel", [(MAX_CLUSTER * CL_ROWS, "qr.k_qr_panel_cluster"), (MAX_CLUSTER * CL_ROWS + 1, "qr.k_qr_panel"),
                                         ("sms", "qr.k_qr_panel"), ("sms+1", "qr.k_qr_panel")])
def test_qr_panel_kernel_at_the_switch(eng, num_sms, rows, kernel):
    if rows in ("sms", "sms+1"):
        rows = num_sms * CL_ROWS + (rows == "sms+1")     # widest grid with shared-memory slabs / first with global ones
    rng = np.random.default_rng(rows)
    psi = crand(rng, rows, 1, 33)
    with launched(eng) as labels:
        Ad, sd = eng.qr_shift("A", eng.to_device(psi))
    if kernel == "qr.k_qr_panel_cluster" and kernel not in labels:
        pytest.skip("no 16-CTA cluster of k_qr_panel_cluster is schedulable on this device")
    assert kernel in labels
    A, s = orc.shift_qr(psi)
    np.testing.assert_allclose(Ad.cpu().numpy(), A, atol=1e-12)   # unique Q, R for Gaussian input: elementwise
    np.testing.assert_allclose(sd.cpu().numpy(), s, atol=1e-12 * np.abs(s).max())


def _mixed_path_qr(eng, psi):
    with launched(eng) as labels:
        Ad, sd = eng.qr_shift("A", eng.to_device(psi))
    if "qr.k_qr_panel_cluster" not in labels:
        pytest.skip("no 16-CTA cluster of k_qr_panel_cluster is schedulable on this device")
    # panels 0-3 have 4200 ... 4104 rows (cooperative), panels 4-6 4072 ... 4008 (cluster)
    assert "qr.k_qr_panel" in labels
    return Ad.cpu().numpy(), sd.cpu().numpy()


def test_qr_mixed_panel_kernels(eng):
    psi = crand(np.random.default_rng(420), 420, 10, 200)
    Ad, sd = _mixed_path_qr(eng, psi)
    A, s = orc.shift_qr(psi)
    np.testing.assert_allclose(Ad, A, atol=1e-12)
    np.testing.assert_allclose(sd, s, atol=1e-12 * np.abs(s).max())
    Q = Ad.reshape(4200, 200)
    assert orth(Q) <= 1e-13
    assert np.linalg.norm(Q @ sd - psi.reshape(4200, 200)) <= 1e-13 * np.linalg.norm(psi)


def test_qr_mixed_panel_kernels_lapack_completion(eng):
    """Exactly-zero columns 30-40 cross the panel edge at 32: tau = 0 reflectors in the cooperative panels, and the
    null-space completion must still be LAPACK's."""
    psi = crand(np.random.default_rng(421), 420, 10, 200)
    psi[:, :, 30:41] = 0.0
    Ad, sd = _mixed_path_qr(eng, psi)
    A, s = orc.shift_qr(psi)
    np.testing.assert_allclose(Ad, A, atol=1e-13)
    np.testing.assert_allclose(sd, s, atol=1e-13 * np.abs(s).max())


def test_qr_cooperative_tiny_tails(eng):
    """5000-row version of test_svd_and_qr_denormal_directions: the zlarfg tiny-tail branch of k_qr_panel."""
    rng = np.random.default_rng(5000)
    psi = (crand(rng, 6, 5000) * np.array([1.0, 2e-13, 8e-18, 7e-157, 0.0, 0.0])[:, None]).reshape(6, 4, 1250)
    with launched(eng) as labels:
        B, sig = eng.qr_shift("B", eng.to_device(psi))
    assert "qr.k_qr_panel" in labels
    Bm = B.cpu().numpy().reshape(6, 5000)
    np.testing.assert_allclose(Bm @ Bm.conj().T, np.eye(6), atol=1e-13)
    np.testing.assert_allclose(np.tensordot(sig.cpu().numpy(), B.cpu().numpy(), axes=(1, 0)), psi, atol=1e-15)


# ---------------------------------------------------------------------------------------------------------------------
# 3. SVD: blocked against plain Jacobi, and relative accuracy against a 40-digit reference
def svd_kernel(m, n):
    """The kernel svd_exec picks (B200: the blocked kernel is always schedulable)."""
    for b in (16, 8, 4, 2):
        if 2 * b * m * 16 <= SVD_SMEM:
            return "svd.k_jacobi_svd_blocked" if n <= 2 * b else "svd.k_jacobi_svd"
    return "svd.k_jacobi_svd"


@pytest.mark.parametrize("m,n", [(320, 32), (321, 32), (640, 16), (641, 16), (1280, 8), (1281, 8), (2560, 4), (2561, 4),
                                 (300, 17), (99, 33)])
def test_svd_blocked_plain_switch(eng, m, n):
    rng = np.random.default_rng(m * 100 + n)
    M = crand(rng, m, n)
    with launched(eng) as labels:
        U, s, Vh = eng.svd(eng.to_device(M))
    kernel = svd_kernel(m, n)
    assert kernel in labels
    assert ({"svd.k_jacobi_svd_blocked", "svd.k_jacobi_svd"} - {kernel}).isdisjoint(labels)
    U, Vh = U.cpu().numpy(), Vh.cpu().numpy()
    s_ref = np.linalg.svd(M, compute_uv=False)
    assert orth(U) < 20 * np.sqrt(m) * EPS                   # one-sided Jacobi: ~ sqrt(m) EPS per column pair
    assert orth(Vh.conj().T) < 20 * n * EPS                  # product of O(n^2) exact-ish rotations per sweep
    assert np.abs((U * s[None, :]) @ Vh - M).max() < 20 * np.sqrt(m) * EPS * s_ref[0]
    assert np.abs(s - s_ref).max() <= 1e-12 * s_ref[0]       # LAPACK: absolute accuracy ~ n EPS s_max


@pytest.mark.parametrize("m,n", [(24, 8), (40, 17), (64, 33)])
def test_svd_relative_accuracy_graded(eng, m, n):
    """Column-graded A = B diag(10^(-12 j/(n-1))) with kappa(B) = 10: one-sided Jacobi determines every singular value
    to ~ kappa(B) n EPS relative (Demmel-Veselic), which LAPACK's bidiagonal SVD does not, so the reference is mpmath at
    40 digits.  Bar: 1e-11 relative for every value (~ 45000 EPS, well above kappa(B) n sqrt(m) EPS)."""
    import mpmath

    rng = np.random.default_rng(m + n)
    Q1, _ = np.linalg.qr(crand(rng, m, n))
    Q2, _ = np.linalg.qr(crand(rng, n, n))
    B = (Q1 * np.linspace(1.0, 10.0, n)[None, :]) @ Q2.conj().T
    A = B * 10.0 ** (-12.0 * np.arange(n) / (n - 1))[None, :]
    with launched(eng) as labels:
        _, s, _ = eng.svd(eng.to_device(A))
    assert svd_kernel(m, n) in labels
    with mpmath.workdps(40):
        s_ref = mpmath.svd_c(mpmath.matrix(A.tolist()), compute_uv=False)
        s_ref = np.array(sorted((float(x) for x in s_ref), reverse=True))
    assert s_ref[-1] < 1e-11 * s_ref[0]
    np.testing.assert_array_less(np.abs(s - s_ref), 1e-11 * s_ref)


def _pinv_diag_input(rcond):
    cut = rcond * 5.0                                  # the device's cut: rcond * max|d|, max|d| = |3 + 4i| = 5 exactly
    # |x| of a real or imaginary x is exact, and so is sqrt(x^2): the three entries sit at, above and below the cut
    d = np.array([3 + 4j, -2j, 0.7, 1j * cut, 1j * np.nextafter(cut, np.inf), -np.nextafter(cut, 0.0), 0.0])
    return np.diag(d).astype(np.complex128), d


def test_pinv_diagonal_at_the_cut(eng):
    rcond = 1e-3
    X, d = _pinv_diag_input(rcond)
    with launched(eng) as labels:
        got = eng.pinv(eng.to_device(X), rcond).cpu().numpy()
    assert not labels & {"svd.k_jacobi_svd_blocked", "svd.k_jacobi_svd"}      # the diagonal shortcut
    keep = np.array([1, 1, 1, 0, 1, 0, 0], dtype=bool)                         # strictly above the cut, as numpy
    expect = np.diag(np.where(keep, 1.0 / np.where(keep, d, 1.0), 0.0))
    np.testing.assert_array_equal(got != 0, expect != 0)
    np.testing.assert_allclose(got, expect, rtol=10 * EPS, atol=0)            # one complex division per entry
    np.testing.assert_allclose(got, np.linalg.pinv(X, rcond=rcond), rtol=50 * EPS, atol=0)   # LAPACK: SVD + product


def test_pinv_almost_diagonal_takes_the_svd(eng):
    rcond = 1e-3
    X, _ = _pinv_diag_input(rcond)
    X[0, 5] = 1e-300
    with launched(eng) as labels:
        got = eng.pinv(eng.to_device(X), rcond).cpu().numpy()
    assert labels & {"svd.k_jacobi_svd_blocked", "svd.k_jacobi_svd"}
    ref = np.linalg.pinv(X, rcond=rcond)
    assert np.abs(got[[3, 5, 6], [3, 5, 6]]).max() < 1e-200                      # the entries at and below the cut stay cut
    np.testing.assert_allclose(got, ref, rtol=0, atol=20 * 7 * EPS * np.abs(ref).max())   # SVD + GEMM: ~ n EPS


@pytest.mark.parametrize("x", [0.37 - 1.2j, 0.0 + 0.0j])
def test_pinv_one_by_one(eng, x):
    X = np.array([[x]])
    np.testing.assert_allclose(eng.pinv(eng.to_device(X), 1e-13).cpu().numpy(), np.linalg.pinv(X, rcond=1e-13),
                               rtol=10 * EPS, atol=0)   # one complex division


# ---------------------------------------------------------------------------------------------------------------------
# 4. Lanczos: fused against unfused step on one kind of operator, H = L (x) W (x) R
def _heff(rng, Dl, d, Dr):
    return hermitian(rng, Dl).reshape(Dl, 1, Dl), hermitian(rng, d).reshape(1, d, d, 1), hermitian(rng, Dr).reshape(Dr, 1, Dr)


def _run_sil(eng, L, W, R, psi, scale, n_hist, cn):
    core = orc.SiteCore((0, 1, 2), 1, W, False, False)
    N = psi.size
    ref, nref = orc.sil_reference(scale, lambda v: orc.heff_term(L, core, R, v), psi, 1e-9, last_niter=n_hist,
                                  conserve_norm=cn)
    _, n_warm = orc.krylov_warmup(N, n_hist)
    psid = eng.to_device(psi)
    with launched(eng) as labels:
        niter = eng.krylov_expm("lanczos", scale, 1e-9, n_warm, cn, psid,
                                hterms=[(eng.to_device(L), eng.upload_core(W), eng.to_device(R), 1.0)])
    kernel = "vec.k_lanczos_step_small" if N <= FUSED_MAX_N else "vec.k_lanczos_update"
    assert kernel in labels
    assert ({"vec.k_lanczos_step_small", "vec.k_lanczos_update"} - {kernel}).isdisjoint(labels)
    return psid.cpu().numpy(), niter, ref, nref


@pytest.mark.parametrize("Dl,d,Dr", [(32, 32, 32), (9, 11, 331), (7, 31, 151), (1, 1, 1), (7, 73, 1), (17, 241, 1)])
@pytest.mark.parametrize("cn", [True, False])
@pytest.mark.parametrize("n_hist", [0, 8])
def test_lanczos_fused_switch(eng, Dl, d, Dr, cn, n_hist):
    """N = 32768 (fused), 32769 and 32767 on both sides, and small N = 1, 511, 4097."""
    rng = np.random.default_rng(Dl * 10000 + d * 100 + Dr)
    L, W, R = _heff(rng, Dl, d, Dr)
    psi = crand(rng, Dl, d, Dr)
    psi *= (1.0 if cn else 1.7) / np.linalg.norm(psi)
    got, niter, ref, nref = _run_sil(eng, L, W, R, psi, -0.3j, n_hist, cn)
    assert niter == nref
    assert relerr(got, ref) < 1e-12      # ~ niter x N-term inner products: sqrt(N) niter EPS << 1e-12


@pytest.mark.parametrize("Dl,d,Dr", [(32, 32, 32), (9, 11, 331)])
def test_lanczos_breakdown_in_invariant_subspace(eng, Dl, d, Dr):
    """A breakdown (beta < 1e-12) inside the warm-up (8 steps), so the Ritz step of the breakdown is the first one
    computed.  The reference's recurrence takes alpha_l = <v0|H v_l>, not <v_l|H v_l>: its basis is not orthogonal and it
    does not break down on a k > 1 dimensional invariant subspace, only on an eigenvector (beta_0 = 0, niter = 1)."""
    rng = np.random.default_rng(Dl + d + Dr)
    # real symmetric factors: the invariant subspace does not depend on which index of L / W / R the contraction sums
    Ul, _ = np.linalg.qr(rng.standard_normal((Dl, Dl)))
    L = ((Ul * np.linspace(-1.0, 1.0, Dl)[None, :]) @ Ul.T).reshape(Dl, 1, Dl).astype(np.complex128)
    Wm, Rm = hermitian(rng, d).real.astype(np.complex128), hermitian(rng, Dr).real.astype(np.complex128)
    x = np.linalg.eigh(Wm)[1][:, 0]
    y = np.linalg.eigh(Rm)[1][:, -1]
    psi = (0.6 - 0.8j) * np.einsum("a,b,c->abc", Ul[:, 3], x, y)
    psi /= np.linalg.norm(psi)
    got, niter, ref, nref = _run_sil(eng, L, Wm.reshape(1, d, d, 1), Rm.reshape(Dr, 1, Dr), psi, -0.5j, 10, True)
    assert nref == 1 and niter == 1
    assert relerr(got, ref) < 1e-12


# ---------------------------------------------------------------------------------------------------------------------
# 5. bra != ket: overlap_site with different bond dimensions, and Simulator.operate on the device
@pytest.mark.parametrize("conj", [False, True])
def test_overlap_site_bra_ket_dimensions(eng, conj):
    rng = np.random.default_rng(31 + conj)
    Dlb, Dlk, d, Drb, Drk = 5, 7, 3, 6, 4
    bra, ket, blk = crand(rng, Dlb, d, Drb), crand(rng, Dlk, d, Drk), crand(rng, Dlb, Dlk)
    ref = np.einsum("abc,abk->ck", np.conj(bra) if conj else bra, np.einsum("ibk,ai->abk", ket, blk))
    out = eng.overlap_site(eng.to_device(bra), eng.to_device(ket), eng.to_device(blk), conj)
    assert relerr(out.cpu().numpy(), ref) < 1e-13


@pytest.mark.parametrize("tag", ["prod", "prop"])
def test_operate_on_device_matches_reference(tag, tmp_path, monkeypatch):
    """tests/test_operate_cpu.py::test_operate_matches_reference with the device Engine: apply_dipole's environments
    have bra != ket."""
    import os

    import pytdscf_b200 as tb
    from tests.golden_io import GOLDEN_DIR
    from tests.test_operate_cpu import dense, operator_model

    z = dict(np.load(os.path.join(GOLDEN_DIR, "operate.npz")))
    model, _ = operator_model(z)
    monkeypatch.chdir(tmp_path)
    sim = tb.Simulator("operate_" + tag, model, backend="cuda", device=0, verbose=0)
    init = [z[f"{tag}_init{i}"] for i in range(4)]
    sim.set_initial_mps(init, [str(g) for g in z[f"{tag}_init_gauges"]])
    norm, wf = sim.operate(maxstep=10)
    assert abs(norm - float(z[f"{tag}_norm"])) < 1e-10 * float(z[f"{tag}_norm"])
    got = wf.ci_coef.to_numpy()
    final = [z[f"{tag}_final{i}"] for i in range(4)]
    assert [c.shape for c in got] == [c.shape for c in final]
    assert [s.gauge for s in wf.ci_coef.sites] == [str(g) for g in z[f"{tag}_final_gauges"]]
    np.testing.assert_allclose(dense(got), dense(final), rtol=0, atol=1e-10)
