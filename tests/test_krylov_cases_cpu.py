"""CPU checks of the premises behind tests/test_gpu_krylov.py, run on the oracle: a broken case builder or reference fails
here without a GPU."""
import mpmath
import numpy as np
import pytest
import scipy.linalg

from oracle import tdvp_oracle as orc
from tests import krylov_cases as kc

EPS = kc.EPS


# The premise that matters is the device's arithmetic: it divides by beta part by part, exactly, so its basis stays at
# the unit vectors bit for bit.  ``kc.*_basis`` emulate that order of operations and must give V = I exactly.  The
# oracle's basis only stays near them: NumPy's in-place w /= beta divides complex by real as complex by complex, which
# can leave 1 - 2^-53 instead of 1, and that drift grows to ~1e-12 by n = 20; from the oracle only niter is checked.


@pytest.mark.parametrize("n", [1, 2, 3, 7, 19, 20])
@pytest.mark.parametrize("family", sorted(kc.HESS_FAMILIES))
def test_exact_basis_arnoldi(family, n):
    H = kc.HESS_FAMILIES[family](n)
    assert np.allclose(np.tril(H, -2), 0) and np.all(np.diag(H, -1).real > 0) and np.all(np.diag(H, -1).imag == 0)
    _, niter = orc.sia_reference(-3j, lambda v: H @ v, kc.e0(n), 0.0, conserve_norm=False)
    assert niter == n
    V, beta = kc.arnoldi_basis(H)
    assert np.array_equal(V, np.eye(n)) and beta[-1] == 0.0


@pytest.mark.parametrize("n", [2, 12, 20])
@pytest.mark.parametrize("im_a0", [0.0, 0.9e-10, 1.1e-10, 0.3])
def test_exact_basis_lanczos_ref(n, im_a0):
    T = kc.lanczos_ref_tridiag(n, im_a0)
    _, niter = orc.sil_reference(-3j, lambda v: T @ v, kc.e0(n), 0.0, conserve_norm=False)
    assert niter == n
    V, alpha, beta = kc.lanczos_ref_basis(T)
    assert np.array_equal(V, np.eye(n)) and beta[-1] == 0.0
    # the tridiagonal the solver builds from (alpha, beta) is T itself
    assert np.array_equal(np.diag(alpha) + np.diag(beta[:-1], 1) + np.diag(beta[:-1], -1), T)


@pytest.mark.parametrize("n", [2, 33, 66, 200])
@pytest.mark.parametrize("family", ["random", "laplacian-", "laplacian+", "graded", "negdef", "scaled1e6", "scaled1e-6"])
def test_exact_basis_textbook_lanczos(family, n):
    a, b = kc.tridiag_family(family, n)
    T = kc.tridiag_dense(a, b).astype(np.complex128)
    V, _, beta = kc.textbook_lanczos_basis(a, b)
    assert V.shape == (n, n) and beta[-1] == 0.0
    assert np.array_equal(np.abs(V), np.eye(n))
    if family.startswith("laplacian"):
        # off-diagonals +-1: NumPy's w /= beta is exact here too, so the oracle runs the same recurrence (elsewhere its
        # complex-by-real division leaves rounding in the last step and it takes one more step than the device)
        _, niter = orc.lanczos_ground_state(lambda v: T @ v, kc.e0(n), thresh=0.0)
        assert niter == n


def test_mp_expm_matches_scipy_for_small_norms():
    rng = np.random.default_rng(5)
    for n in (1, 2, 7, 20):
        for A in (kc.hess_random(n), kc.hess_hermitian(n), kc.hess_nonnormal(n), np.triu(kc.crand(rng, n, n), -1)):
            A = A / max(kc.norm1(A), 1.0)
            ref = scipy.linalg.expm(A)[:, 0]
            got = kc.mp_expm_e0(A)
            assert np.linalg.norm(got - ref) <= 1e-14 * np.linalg.norm(ref)


def test_expm_kappa():
    """kappa of a scalar a is |a|, also where exp(a) ~ 1e243 squares to an overflow; a small Hermitian exponent is well
    conditioned."""
    for a in (-3000j, 0.3 - 2j, -20.0, 560.0, 560.0 - 3000j):
        assert abs(kc.expm_kappa(np.array([[a]])) - abs(a)) < 1e-12 * abs(a)
    assert kc.expm_kappa(-0.05j * kc.hess_hermitian(7)) < 2


def test_mp_eigenvalue_matches_eigsy():
    for family in ("random", "graded", "laplacian-"):
        a, b = kc.tridiag_family(family, 12)
        with mpmath.workdps(40):
            E, _ = mpmath.eigsy(mpmath.matrix(kc.tridiag_dense(a, b).tolist()))
            ev = sorted(float(x) for x in E)
        nT = np.abs(ev).max()
        assert abs(kc.mp_extreme_eigenvalue(a, b, 0) - ev[0]) <= 2 * EPS * nT
        assert abs(kc.mp_extreme_eigenvalue(a, b, 1) - ev[-1]) <= 2 * EPS * nT


@pytest.mark.parametrize("kind", ["arnoldi", "lanczos"])
@pytest.mark.parametrize("ks,last_niter", [((2, 2, 1), 10), ((3, 3, 1), 10), ((2, 5, 1), 10), ((1, 1, 1), 0),
                                           ((2, 1, 1), 0), ((2, 5, 2), 10)])
def test_kron_breakdown_niter(kind, ks, last_niter):
    """Arnoldi breaks down at l = k - 1 on the k-dimensional invariant subspace; the reference Lanczos only on k = 1."""
    dims = (16, 16, 16)
    Lm, Wm, Rm, psi, P, Ak, c = kc.kron_breakdown_case(dims, ks)
    k = int(np.prod(ks))
    assert np.linalg.norm(P.conj().T @ P - np.eye(k)) < 1e-13
    mv = kc.kron_matvec(Lm, Wm, Rm)
    ref = (P @ (scipy.linalg.expm((0.2 - 1j) * Ak) @ c)).reshape(dims)
    if kind == "arnoldi":
        got, niter = orc.sia_reference(0.2 - 1j, mv, psi, 0.0, last_niter=last_niter, conserve_norm=False)
        assert niter == k
        assert np.abs(got - ref).max() <= 1e-12 * np.abs(ref).max()
    elif k == 1:
        got, niter = orc.sil_reference(0.2 - 1j, mv, psi, 1e-9, last_niter=last_niter, conserve_norm=False)
        assert niter == 1
        assert np.abs(got - ref).max() <= 1e-12 * np.abs(ref).max()


def test_small_expm_hook():
    """The optional small step replaces only the eigen-decomposition: with an accurate exponential the result stays within
    rounding of the reference arithmetic on a well-conditioned operator, and niter is unchanged."""
    rng = np.random.default_rng(9)
    n = 30
    H = kc.crand(rng, n, n)
    H = (H + H.conj().T) / (2 * np.sqrt(n))
    x = kc.crand(rng, n)
    for solver in (orc.sil_reference, orc.sia_reference):
        a, na = solver(-0.5j, lambda v: H @ v, x, 1e-9, conserve_norm=False)
        b, nb = solver(-0.5j, lambda v: H @ v, x, 1e-9, conserve_norm=False, small_expm=kc.mp_expm_e0)
        assert na == nb
        assert np.abs(a - b).max() < 1e-12 * np.abs(a).max()
