"""GPU tests of the Krylov solvers of csrc/krylov.cu beyond the reference goldens: the small matrix exponential and the
tridiagonal eigenvector kernels against mpmath, and every stopping branch of the Arnoldi, reference-Lanczos and textbook
Lanczos loops.

  A  k_krylov_small_expm, Hessenberg mode: Arnoldi on exact-basis operators (tests/krylov_cases.py), so the Ritz step
     exponentiates a Hessenberg matrix the test chose; scales from -0.05j to -3000j (up to 13 squarings), real and
     complex; against mpmath.expm at 60 digits, bar 32 n EPS max(1, kappa)
  B  the same kernel in tridiagonal mode, with Im a_0 on both sides of the 1e-10 "alpha is real" threshold
  C  general operators against the oracle whose small step is mpmath's exponential
  D  Arnoldi breakdown at every position of the loop: inside the warm-up, at the first checked iteration (whose Ritz step
     runs on the side stream), after it, at the last vector; eigenvector inputs and exact beta = 0 for both kinds
  E  tdvp_set_krylov_size (adaptive bond growth) with the warm-up clamped to the original size; the override is one-shot
  F  the error contract: not converged in 20 vectors, zero norm, NaN
  G  lanczos_eigvec: exact-basis tridiagonals through every basis growth, root 0 and 1, breakdown part-way, a general
     operator that needs more than 64 vectors, and the 3000-vector cap

Every group reports its largest error / bar ratio at the end of the module (visible with -s).
"""
import time

import numpy as np
import pytest
import scipy.linalg

from oracle import tdvp_oracle as orc
from tests import krylov_cases as kc

pytestmark = pytest.mark.gpu

EPS = kc.EPS
SCALE_IDS = [str(s) for s in kc.EXPM_SCALES]


@pytest.fixture(scope="module")
def eng():
    from pytdscf_b200._engine import Engine

    e = Engine(0)
    yield e
    e.close()


_RATIOS: dict = {}


@pytest.fixture(scope="module", autouse=True)
def report():
    t0 = time.time()
    yield
    print("\n[krylov] largest error / bar per group:")
    for g in sorted(_RATIOS):
        print(f"[krylov]   {g}: {_RATIOS[g]:.3g}")
    print(f"[krylov] module time {time.time() - t0:.1f} s")


def note(group, err, bar):
    _RATIOS[group] = max(_RATIOS.get(group, 0.0), err / bar)
    return err <= bar


def dense_terms(eng, M):
    """A dense n x n operator as one H_eff term: (n, 1, n) left block, identity core and right block."""
    n = M.shape[0]
    return [(eng.to_device(M.reshape(n, 1, n)), None, None, 1.0)]


def kron_terms(eng, Lm, Wm, Rm):
    Dl, d, Dr = Lm.shape[0], Wm.shape[0], Rm.shape[0]
    return [(eng.to_device(Lm.reshape(Dl, 1, Dl)), eng.upload_core(Wm.reshape(1, d, d, 1)),
             eng.to_device(Rm.reshape(Dr, 1, Dr)), 1.0)]


def rel(got, want):
    s = np.abs(want).max()
    return np.linalg.norm((got - want) / s) / np.linalg.norm(want / s)


def out_of_range(ref):
    """True when the exponential is not finite in double or above 1e250: complex-eigenvalue operators at imaginary
    scales grow like exp(3000 |Im lambda|), and those cases are left out like the large real scales."""
    return not (np.all(np.isfinite(ref)) and np.abs(ref).max() <= kc.EXPM_MAX)


def underflows(ref):
    """True when every entry of the exponential is below 1e-250 in magnitude (e.g. exp(-2695) for n = 1 at scale -3000j):
    double cannot hold it to relative accuracy, and its normalised column is 0 / 0 in the reference as well."""
    return np.abs(ref).max() < 1.0 / kc.EXPM_MAX


def norm_overflows(ref):
    """True when sum |y|^2 overflows (|y| above ~1e154).  The normalised column y / |y| of conserve_norm is then not
    formed by the device nor by the reference (both take |y| as the square root of that sum), so only the raw column is
    compared there."""
    return np.abs(ref).max() > 1e150


def unit_psi(eng, n):
    return eng.to_device(kc.e0(n).reshape(n, 1, 1))


# ---------------------------------------------------------------------------------------------------------------------
# A. the small exponential, Hessenberg mode
@pytest.mark.parametrize("scale", kc.EXPM_SCALES, ids=SCALE_IDS)
@pytest.mark.parametrize("n", [1, 2, 3, 7, 19, 20])
@pytest.mark.parametrize("family", sorted(kc.HESS_FAMILIES))
def test_small_expm_hessenberg(eng, family, n, scale):
    H = kc.HESS_FAMILIES[family](n)
    A = scale * H
    ref = kc.mp_expm_e0(A)
    if out_of_range(ref):
        pytest.skip("exponential above 1e250")
    terms = dense_terms(eng, H)
    if underflows(ref):
        # no relative error to measure: the raw column must be finite and underflow as well
        for n_hist in (0, 10):
            _, n_warm = orc.krylov_warmup(n, n_hist)
            psi = unit_psi(eng, n)
            assert eng.krylov_expm("arnoldi", scale, 0.0, n_warm, False, psi, hterms=terms) == n
            got = psi.cpu().numpy()
            assert np.all(np.isfinite(got)) and np.abs(got).max() < 1.0 / kc.EXPM_MAX
        return
    bar = kc.expm_bar(A)
    for n_hist in (0, 10):
        _, n_warm = orc.krylov_warmup(n, n_hist)
        for cn in (False, True):
            if cn and norm_overflows(ref):
                continue
            psi = unit_psi(eng, n)
            niter = eng.krylov_expm("arnoldi", scale, 0.0, n_warm, cn, psi, hterms=terms)
            assert niter == n
            want = ref / np.linalg.norm(ref) if cn else ref
            err = rel(psi.cpu().numpy().reshape(-1), want)
            assert note("A", err, bar), (n_hist, cn, err, bar)


# ---------------------------------------------------------------------------------------------------------------------
# B. the small exponential, tridiagonal mode
@pytest.mark.parametrize("scale", kc.EXPM_SCALES, ids=SCALE_IDS)
@pytest.mark.parametrize("im_a0", [0.0, 0.9e-10, 1.1e-10, 0.3])
@pytest.mark.parametrize("n", [2, 12, 20])
def test_small_expm_tridiagonal(eng, n, im_a0, scale):
    """While every |Im alpha| <= 1e-10 the reference exponentiates the real part (eigh_tridiagonal(np.real(alpha))); above
    that the complex matrix.  At scale -3j the two differ by ~3e-10 for Im a_0 = 1e-10."""
    T = kc.lanczos_ref_tridiag(n, im_a0)
    A = scale * (T.real.astype(np.complex128) if im_a0 <= 1e-10 else T)
    ref = kc.mp_expm_e0(A)
    if out_of_range(ref):
        pytest.skip("exponential above 1e250")
    bar = kc.expm_bar(A)
    terms = dense_terms(eng, T)
    for cn in (False, True):
        if cn and norm_overflows(ref):
            continue
        psi = unit_psi(eng, n)
        niter = eng.krylov_expm("lanczos", scale, 0.0, 0, cn, psi, hterms=terms)
        assert niter == n
        want = ref / np.linalg.norm(ref) if cn else ref
        err = rel(psi.cpu().numpy().reshape(-1), want)
        assert note("B", err, bar), (cn, err, bar)


# ---------------------------------------------------------------------------------------------------------------------
# C. general operators, oracle with an mpmath small step
def _psd(rng, n, width):
    if n == 1:
        return np.full((1, 1), 0.5 * width, dtype=np.complex128)
    X = kc.crand(rng, n, n)
    w, U = np.linalg.eigh((X + X.conj().T) / 2)
    return (U * ((w - w.min()) / (w.max() - w.min()) * width)) @ U.conj().T


def _nonherm(rng, n):
    return kc.crand(rng, n, n) / np.sqrt(2 * n)


def _check_oracle(group, got, niter, ref, nref):
    assert niter == nref
    assert note(group, rel(got, ref), 1e-12)


@pytest.mark.parametrize("scale", [-0.5, -5.0, -50.0, 0.5])
def test_hermitian_heff_relaxation_scales(eng, scale):
    """Imaginary-time steps: real scales, conserve_norm.  The spectrum of H lies in [0, 0.1], so |scale H| <= 5."""
    rng = np.random.default_rng(61)
    Lm, Wm, Rm = _psd(rng, 6, 0.1), _psd(rng, 5, 1.0), _psd(rng, 7, 1.0)
    psi = kc.crand(rng, 6, 5, 7)
    psi /= np.linalg.norm(psi)
    ref, nref = orc.sil_reference(scale, kc.kron_matvec(Lm, Wm, Rm), psi, 1e-9, small_expm=kc.mp_expm_e0)
    psid = eng.to_device(psi)
    niter = eng.krylov_expm("lanczos", scale, 1e-9, 0, True, psid, hterms=kron_terms(eng, Lm, Wm, Rm))
    _check_oracle("C", psid.cpu().numpy(), niter, ref, nref)


@pytest.mark.parametrize("cn", [False, True])
def test_nonhermitian_heff_arnoldi(eng, cn):
    rng = np.random.default_rng(62 + cn)
    Lm, Wm, Rm = _nonherm(rng, 9), _psd(rng, 4, 1.0).astype(np.complex128), _nonherm(rng, 8)
    psi = kc.crand(rng, 9, 4, 8)
    psi *= 1.7 / np.linalg.norm(psi)
    ref, nref = orc.sia_reference(0.2 - 1j, kc.kron_matvec(Lm, Wm, Rm), psi, 1e-9, conserve_norm=cn,
                                  small_expm=kc.mp_expm_e0)
    psid = eng.to_device(psi)
    niter = eng.krylov_expm("arnoldi", 0.2 - 1j, 1e-9, 0, cn, psid, hterms=kron_terms(eng, Lm, Wm, Rm))
    _check_oracle("C", psid.cpu().numpy(), niter, ref, nref)


@pytest.mark.parametrize("kind", ["arnoldi", "lanczos"])
def test_keff_small_expm(eng, kind):
    """K_eff (bond) solves with non-Hermitian blocks through both kinds."""
    D, w = 20, 3
    rng = np.random.default_rng(64)
    L = kc.crand(rng, D, w, D) / np.sqrt(2 * D * w)
    R = kc.crand(rng, D, w, D) / np.sqrt(2 * D * w)
    s = kc.crand(rng, D, D)
    s /= np.linalg.norm(s)
    solver = orc.sia_reference if kind == "arnoldi" else orc.sil_reference
    ref, nref = solver(0.2 - 1j, lambda v: orc.keff_term(L, R, v), s, 1e-9, small_expm=kc.mp_expm_e0)
    sd = eng.to_device(s)
    niter = eng.krylov_expm(kind, 0.2 - 1j, 1e-9, 0, True, sd, kterms=[(eng.to_device(L), eng.to_device(R), 1.0)])
    _check_oracle("C", sd.cpu().numpy(), niter, ref, nref)


# ---------------------------------------------------------------------------------------------------------------------
# D. breakdown at every position
BREAKDOWN_KS = {1: (1, 1, 1), 2: (2, 1, 1), 4: (2, 2, 1), 9: (3, 3, 1), 10: (2, 5, 1), 20: (2, 5, 2)}


@pytest.mark.parametrize("dims", [(16, 16, 16), (40, 25, 40)], ids=["N4096", "N40000"])
@pytest.mark.parametrize("n_warm,k", [(8, 4), (8, 9), (8, 10), (0, 1), (0, 2), (8, 20)])
def test_arnoldi_breakdown_positions(eng, dims, n_warm, k):
    """(8, 4): inside the warm-up.  (8, 9): at the first checked iteration, whose Ritz step runs on the side stream and
    whose breakdown the next read-back replays.  (8, 10): the first ordinary read-back.  (0, 1): at l = 0, itself the
    side-stream position.  (0, 2): the read-back after it.  (8, 20): at the last vector."""
    Lm, Wm, Rm, psi, P, Ak, c = kc.kron_breakdown_case(dims, BREAKDOWN_KS[k])
    scale = 0.2 - 1j
    exact = (P @ (scipy.linalg.expm(scale * Ak) @ c)).reshape(dims)
    ref, nref = orc.sia_reference(scale, kc.kron_matvec(Lm, Wm, Rm), psi, 0.0, last_niter=n_warm + 2 if n_warm else 0,
                                  conserve_norm=False)
    assert nref == k
    psid = eng.to_device(psi)
    niter = eng.krylov_expm("arnoldi", scale, 0.0, n_warm, False, psid, hterms=kron_terms(eng, Lm, Wm, Rm))
    got = psid.cpu().numpy()
    assert niter == k
    assert note("D", np.abs(got - exact).max() / np.abs(exact).max(), 1e-12)
    assert note("D", np.abs(got - ref).max() / np.abs(ref).max(), 1e-12)


@pytest.mark.parametrize("dims", [(32, 32, 32), (9, 11, 331)], ids=["N32768", "N32769"])
@pytest.mark.parametrize("kind", ["arnoldi", "lanczos"])
def test_breakdown_at_the_first_vector(eng, kind, dims):
    """niter = 1 on both sides of the fused-step switch: an eigenvector input (beta_0 at rounding level, n_warm = 0: the
    side-stream position) and a diagonal operator on e_3 (beta_0 exactly 0)."""
    Lm, Wm, Rm, psi, P, Ak, c = kc.kron_breakdown_case(dims, (1, 1, 1))
    scale = 0.2 - 1j
    psid = eng.to_device(psi)
    niter = eng.krylov_expm(kind, scale, 1e-9, 0, False, psid, hterms=kron_terms(eng, Lm, Wm, Rm))
    got = psid.cpu().numpy()
    assert niter == 1 and np.all(np.isfinite(got))
    exact = np.exp(scale * Ak[0, 0]) * psi
    assert note("D", np.abs(got - exact).max() / np.abs(exact).max(), 1e-12)

    rng = np.random.default_rng(70)
    Dl, d, Dr = dims
    dl, dw, dr = rng.uniform(0.5, 1.5, Dl), rng.uniform(0.5, 1.5, d), rng.uniform(0.5, 1.5, Dr)
    x = np.zeros(dims, dtype=np.complex128)
    x.reshape(-1)[3] = 0.8 - 0.6j
    xd = eng.to_device(x)
    niter = eng.krylov_expm(kind, scale, 1e-9, 0, True, xd,
                            hterms=kron_terms(eng, np.diag(dl).astype(complex), np.diag(dw).astype(complex),
                                              np.diag(dr).astype(complex)))
    got = xd.cpu().numpy()
    lam = dl[0] * dw[0] * dr[3]
    assert niter == 1 and np.all(np.isfinite(got))
    assert note("D", np.abs(got - np.exp(scale * lam) * x / abs(np.exp(scale * lam))).max(), 1e-14)


# ---------------------------------------------------------------------------------------------------------------------
# E. Krylov-size override (adaptive bond growth)
def _padded_case(rng, small, big, hermitian):
    """An operator on the zero-extended site tensor, as the adaptive sweep builds it: blocks padded with zeros, psi in the
    original corner."""
    (l, c, r), (Lb, _, Rb) = small, big
    mk = (lambda n: _psd(rng, n, 1.0)) if hermitian else (lambda n: _nonherm(rng, n))
    Lm, Rm = np.zeros((Lb, Lb), complex), np.zeros((Rb, Rb), complex)
    Lm[:l, :l] = mk(l)
    Rm[:r, :r] = mk(r)
    Wm = _psd(rng, c, 1.0).astype(np.complex128)
    psi = np.zeros((Lb, c, Rb), complex)
    psi[:l, :, :r] = kc.crand(rng, l, c, r)
    psi /= np.linalg.norm(psi)
    return Lm, Wm, Rm, psi


@pytest.mark.parametrize("small", [(2, 3, 2), (2, 5, 2), (3, 7, 1)], ids=["Nref12", "Nref20", "Nref21"])
@pytest.mark.parametrize("kind", ["arnoldi", "lanczos"])
def test_krylov_size_override(eng, kind, small):
    """n_hist = 17 gives n_warm = 15 for the padded tensor, which the device clamps to Nref; then a solve without the
    override on the same handle runs with the full size again."""
    rng = np.random.default_rng(80 + small[1])
    big = (5, small[1], 4)
    Lm, Wm, Rm, psi = _padded_case(rng, small, big, kind == "lanczos")
    Nref, N = int(np.prod(small)), int(np.prod(big))
    solver = orc.sia_reference if kind == "arnoldi" else orc.sil_reference
    mv = kc.kron_matvec(Lm, Wm, Rm)
    terms = kron_terms(eng, Lm, Wm, Rm)
    _, n_warm = orc.krylov_warmup(N, 17)
    for override in (Nref, None):
        ref, nref = solver(-0.5j, mv, psi, 1e-9, last_niter=17, maxsize=override)
        psid = eng.to_device(psi)
        niter = eng.krylov_expm(kind, -0.5j, 1e-9, n_warm, True, psid, hterms=terms, size_override=override)
        assert niter == nref, override
        assert note("E", rel(psid.cpu().numpy(), ref), 1e-12), override


# ---------------------------------------------------------------------------------------------------------------------
# F. error contract
def test_not_converged_in_20_vectors(eng):
    from pytdscf_b200._lib import TdvpError

    n = 21
    for kind, M, msg in [("arnoldi", kc.hess_random(n), "Short Iterative Arnoldi is not converged in 20 basis"),
                         ("lanczos", kc.lanczos_ref_tridiag(n), "Short Iterative Lanczos is not converged")]:
        solver = orc.sia_reference if kind == "arnoldi" else orc.sil_reference
        with pytest.raises(ValueError, match=msg):
            solver(-3j, lambda v, M=M: M @ v, kc.e0(n), 0.0)
        psi = unit_psi(eng, n)
        with pytest.raises(TdvpError, match=msg):
            eng.krylov_expm(kind, -3j, 0.0, 0, True, psi, hterms=dense_terms(eng, M))
        assert np.array_equal(psi.cpu().numpy().reshape(-1), kc.e0(n))


@pytest.mark.parametrize("kind", ["arnoldi", "lanczos"])
def test_zero_norm_and_nan(eng, kind):
    from pytdscf_b200._lib import TdvpError

    rng = np.random.default_rng(90)
    n = 30
    M = kc.crand(rng, n, n)
    psi = eng.to_device(np.zeros((n, 1, 1)))
    with pytest.raises(TdvpError, match="Initial psi has zero norm."):
        eng.krylov_expm(kind, -0.5j, 1e-9, 0, False, psi, hterms=dense_terms(eng, M))
    M[3, 5] = np.nan
    for n_warm in (0, 8):
        psi = eng.to_device(kc.crand(rng, n, 1, 1))
        with pytest.raises(TdvpError, match="NaN"):
            eng.krylov_expm(kind, -0.5j, 1e-9, n_warm, True, psi, hterms=dense_terms(eng, M))
    # the handle is usable afterwards
    Mh = kc.crand(rng, n, n)
    Mh = (Mh + Mh.conj().T) / (2 * np.sqrt(n))
    x = kc.crand(rng, n)
    x /= np.linalg.norm(x)
    solver = orc.sia_reference if kind == "arnoldi" else orc.sil_reference
    ref, nref = solver(-0.5j, lambda v: Mh @ v, x, 1e-9)
    psi = eng.to_device(x.reshape(n, 1, 1))
    assert eng.krylov_expm(kind, -0.5j, 1e-9, 0, True, psi, hterms=dense_terms(eng, Mh)) == nref
    assert rel(psi.cpu().numpy().reshape(-1), ref) < 1e-12


def test_lanczos_eigvec_nan(eng):
    from pytdscf_b200._lib import TdvpError

    a, b = kc.tridiag_family("random", 40)
    T = kc.tridiag_dense(a, b).astype(np.complex128)
    T[7, 7] = np.nan
    with pytest.raises(TdvpError, match="NaN"):
        eng.lanczos_eigvec(unit_psi(eng, 40), dense_terms(eng, T), thresh=0.0)


# ---------------------------------------------------------------------------------------------------------------------
# G. textbook Lanczos eigensolver
def _check_eigvec(group, got, a, b, root, check_angle=True):
    """residual |T x - rho x| <= 64 EPS |T|, |rho - lambda| <= 64 EPS |T|, angle <= 64 n EPS |T| / gap (where the gap is
    at least 1e-8 |T|)."""
    n = len(a)
    T = kc.tridiag_dense(a, b)
    lam, v, gap, nT = kc.tridiag_reference(a, b, root)
    x = got.real
    assert np.abs(got.imag).max() == 0.0
    assert abs(np.linalg.norm(x) - 1) <= 1e-14
    assert x[0] > 0                    # positive overlap with the start vector e_0
    rho = x @ T @ x
    tol = 64 * EPS * nT
    assert note(group + " residual", np.linalg.norm(T @ x - rho * x), tol)
    assert note(group + " eigenvalue", abs(rho - lam), tol)
    if check_angle and gap >= 1e-8 * nT:
        ang = np.linalg.norm(x - (v @ x) * v)
        assert note(group + " angle", ang, 64 * n * EPS * nT / gap)


G_NS = [1, 2, 3, 31, 32, 33, 34, 64, 65, 66, 200, 1000]
G_FAMILIES = ["random", "laplacian-", "laplacian+", "graded", "negdef", "scaled1e6", "scaled1e-6"]


@pytest.mark.parametrize("root", [0, 1])
@pytest.mark.parametrize("n", G_NS)
@pytest.mark.parametrize("family", G_FAMILIES)
def test_lanczos_eigvec_exact_basis(eng, family, n, root):
    """The basis starts with room for 32 vectors and doubles (contents preserved, seven pointers rebased) at i = 32, 64,
    ..., so n = 33 / 65 / 200 / 1000 run after one to five growths."""
    a, b = kc.tridiag_family(family, n)
    psi = unit_psi(eng, n)
    niter = eng.lanczos_eigvec(psi, dense_terms(eng, kc.tridiag_dense(a, b).astype(np.complex128)), root=root, thresh=0.0)
    assert niter == n
    _check_eigvec("G", psi.cpu().numpy().reshape(-1), a, b, root)


@pytest.mark.parametrize("root", [0, 1])
def test_lanczos_eigvec_wilkinson(eng, root):
    """W21+: its two largest eigenvalues are ~1e-13 apart, so for root 1 only the residual and eigenvalue are checked."""
    a, b = kc.wilkinson21()
    psi = unit_psi(eng, 21)
    assert eng.lanczos_eigvec(psi, dense_terms(eng, kc.tridiag_dense(a, b).astype(np.complex128)), root=root,
                              thresh=0.0) == 21
    _check_eigvec("G", psi.cpu().numpy().reshape(-1), a, b, root, check_angle=(root == 0))


@pytest.mark.parametrize("root", [0, 1])
@pytest.mark.parametrize("j", [0, 5, 40])
def test_lanczos_eigvec_breakdown(eng, j, root):
    """beta_j = 0 exactly: the solver stops with niter = j + 1 and the eigenvector of the leading block, padded with zeros
    (j = 40 lies after the first growth of the basis)."""
    n = 70
    a, b = kc.tridiag_family("random", n)
    b = b.copy()
    b[j] = 0.0
    psi = unit_psi(eng, n)
    niter = eng.lanczos_eigvec(psi, dense_terms(eng, kc.tridiag_dense(a, b).astype(np.complex128)), root=root, thresh=0.0)
    got = psi.cpu().numpy().reshape(-1)
    assert niter == j + 1
    assert np.all(got[j + 1:] == 0)
    _check_eigvec("G", got[: j + 1], a[: j + 1], b[:j], root)


def _gapped(rng, n, top):
    """Hermitian n x n with eigenvalues in [0, 1.1] and a gap of 0.0005 at the bottom (top = False) or the top."""
    e = np.sort(rng.uniform(0.2, 0.9, n))
    e[0], e[1], e[-2], e[-1] = 0.0, 0.0005, 1.0995, 1.1
    if top:
        e = 1.1 - e[::-1]
    Q, _ = np.linalg.qr(kc.crand(rng, n, n))
    return (Q * e) @ Q.conj().T


@pytest.mark.parametrize("root", [0, 1])
def test_lanczos_eigvec_slow_general_operator(eng, root):
    """H = L (x) 1 (x) 1 + 1 (x) W (x) 1 + 1 (x) 1 (x) R with a gap of 0.0005 at the end of a spectrum of width 3.3: at
    thresh 1e-11 over 64 Lanczos vectors, so the basis grows with the contraction scratch above it.  Root 0 is compared with the
    oracle's textbook Lanczos (whose root indexes the ascending eigenvectors, so only 0 means the same there), both roots
    with eigh."""
    rng = np.random.default_rng(100 + root)
    dims = (12, 6, 12)
    f = [_gapped(rng, n, root == 1) for n in dims]
    eye = [np.eye(n, dtype=np.complex128) for n in dims]
    terms_np = [(f[0], eye[1], eye[2]), (eye[0], f[1], eye[2]), (eye[0], eye[1], f[2])]
    Hd = sum(np.kron(np.kron(L, W), R) for L, W, R in terms_np)
    ws, U = np.linalg.eigh(Hd)
    i = 0 if root == 0 else -1
    x0 = kc.crand(rng, *dims)
    x0 /= np.linalg.norm(x0)
    psi = eng.to_device(x0)
    terms = [t for L, W, R in terms_np for t in kron_terms(eng, L, W, R)]
    niter = eng.lanczos_eigvec(psi, terms, root=root, thresh=1e-11)
    got = psi.cpu().numpy().reshape(-1)
    assert niter > 64
    if root == 0:
        _, nref = orc.lanczos_ground_state(lambda v: (Hd @ v.reshape(-1)).reshape(dims), x0, root=0, thresh=1e-11)
        assert abs(niter - nref) <= 2
    assert abs(abs(np.vdot(U[:, i], got)) - 1) < 1e-9
    assert abs(np.linalg.norm(got) - 1) < 1e-13
    assert np.linalg.norm(Hd @ got - np.vdot(got, Hd @ got) * got) < 1e-7
    assert abs(np.vdot(got, Hd @ got).real - ws[i]) < 1e-9 * max(1.0, abs(ws[i]))


def test_lanczos_eigvec_cap(eng):
    """The reference keeps at most 3000 vectors and takes up to 3001 steps (range(n_iter + 1)): N = 3001 finishes by
    exhaustion at the last of them, N = 3002 raises.  (About 35 s each: the single-thread bisection of k_tridiag_eigvec
    costs O(k) per step for every k up to 3000.)"""
    from pytdscf_b200._lib import TdvpError

    t0 = time.time()
    for n, ok in [(3001, True), (3002, False)]:
        a, b = kc.tridiag_family("random", n)
        psi = unit_psi(eng, n)
        terms = dense_terms(eng, kc.tridiag_dense(a, b).astype(np.complex128))
        if ok:
            assert eng.lanczos_eigvec(psi, terms, thresh=0.0) == n
            _check_eigvec("G cap", psi.cpu().numpy().reshape(-1), a, b, 0)
        else:
            with pytest.raises(TdvpError, match="Lanczos Diagonalization is not converged in 3000 basis"):
                eng.lanczos_eigvec(psi, terms, thresh=0.0)
    print(f"\n[krylov] cap test: {time.time() - t0:.1f} s")
