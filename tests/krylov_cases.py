"""Case builders and high-precision references for the Krylov solvers of csrc/krylov.cu (tests/test_gpu_krylov.py and
tests/test_krylov_cases_cpu.py).

Exact-basis operators.  The small matrix kernels (k_krylov_small_expm, k_tridiag_eigvec) have no entry point of their own.
They are reached through operators for which the recurrence keeps the Krylov basis at the unit vectors, V = I, starting
from psi = e_0: then every inner product and every vector update has exactly one nonzero term, and the small matrix the
kernel receives is a matrix the test chose.
  * Arnoldi: any upper Hessenberg H with a real positive subdiagonal; the Hessenberg block is H itself.
  * reference Lanczos (alpha_l = <v_0|H v_l>): the tridiagonal with diagonal (a_0, b_0, 0, ..., 0) and off-diagonals b_l > 0;
    a_0 may be complex.  The block the kernel builds from (alpha, beta) is that matrix again.
  * textbook Lanczos (lanczos_eigvec): any real symmetric tridiagonal with nonzero off-diagonals.  Negative off-diagonals
    flip the sign of the next basis vector, which is still exact; the solver's answer is the eigenvector of the matrix given.
Each is passed as a dense (n, 1, n) left block with identity core and right block.
"""
from __future__ import annotations

import functools

import mpmath
import numpy as np
import scipy.linalg

EPS = 2.220446049250313e-16
EXPM_DPS = 60
EIG_DPS = 40


def crand(rng, *shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / np.sqrt(2)


def e0(n):
    v = np.zeros(n, dtype=np.complex128)
    v[0] = 1.0
    return v


def rdiv(w, b):
    """w / b for a real b as the device computes it, part by part (NumPy divides complex by real as complex by complex,
    which is not exact: (x + 0j) / x can be 1 - 2^-53)."""
    return (w.real / b) + 1j * (w.imag / b)


def norm1(A):
    return float(np.abs(A).sum(axis=0).max())


# ---------------------------------------------------------------------------------------------------------------------
# matrix exponential: mpmath reference and a condition estimate
def _key(A):
    A = np.ascontiguousarray(A, dtype=np.complex128)
    return A.shape, A.tobytes()


@functools.lru_cache(maxsize=None)
def _mp_expm_col(shape, buf, dps):
    A = np.frombuffer(buf, dtype=np.complex128).reshape(shape)
    with mpmath.workdps(dps):
        E = mpmath.expm(mpmath.matrix(A.tolist()))
        return np.array([complex(E[i, 0]) for i in range(shape[0])])


def mp_expm_e0(A, dps=EXPM_DPS):
    """expm(A)[:, 0] from mpmath at ``dps`` digits (A is taken exactly as stored in double)."""
    return _mp_expm_col(*_key(A), dps).copy()


@functools.lru_cache(maxsize=None)
def _expm_kappa(shape, buf):
    A = np.frombuffer(buf, dtype=np.complex128).reshape(shape)
    n = shape[0]
    f = scipy.linalg.expm(A)[:, 0]
    nA = np.linalg.norm(A)
    m = np.abs(f).max() if np.all(np.isfinite(f)) else 0.0
    if n == 0 or nA == 0.0 or m == 0.0:
        return 1.0
    # f and the derivative are divided by max |f| before any norm: the exponentials tested reach 1e250, whose squares
    # overflow
    nf = np.linalg.norm(f / m)
    rng = np.random.default_rng(n)
    dirs = [A / nA]
    for _ in range(3):
        E = np.triu(crand(rng, n, n), -1)
        dirs.append(E / np.linalg.norm(E))
    best = 1.0
    for E in dirs:
        L = scipy.linalg.expm_frechet(A, E, compute_expm=False)
        k = np.linalg.norm(L[:, 0] / m) * nA / nf
        if not np.isfinite(k):
            raise FloatingPointError("condition estimate is not finite")
        best = max(best, k)
    return best


def expm_kappa(A):
    """Relative condition number of A -> expm(A) e_0, estimated from the Frechet derivative along A / |A| and three random
    Hessenberg directions (the largest of the four, at least 1)."""
    return _expm_kappa(*_key(A))


def expm_bar(A):
    """Relative error bar of a computed expm(A) e_0: 32 n EPS max(1, kappa)."""
    return 32 * A.shape[0] * EPS * max(1.0, expm_kappa(A))


# ---------------------------------------------------------------------------------------------------------------------
# A. Hessenberg families (|.|_1 = 1, real positive subdiagonal)
def hess_random(n, seed=0):
    rng = np.random.default_rng(1000 + 17 * n + seed)
    H = np.triu(crand(rng, n, n), -1)
    for i in range(n - 1):
        H[i + 1, i] = abs(H[i + 1, i]) + 0.1
    return H / norm1(H)


def hess_hermitian(n, seed=0):
    rng = np.random.default_rng(2000 + 17 * n + seed)
    a = rng.standard_normal(n)
    b = rng.uniform(0.1, 1.0, n - 1)
    T = (np.diag(a) + np.diag(b, 1) + np.diag(b, -1)).astype(np.complex128)
    return T / norm1(T)


def hess_nonnormal(n, seed=0):
    """-I + 0.1 (subdiagonal) + 30 (strict upper triangle): far from normal, eigenvalues all -1."""
    H = -np.eye(n, dtype=np.complex128) + 0.1 * np.eye(n, k=-1) + 30.0 * np.triu(np.ones((n, n)), 1)
    return H / norm1(H)


HESS_FAMILIES = {"random": hess_random, "hermitian": hess_hermitian, "nonnormal": hess_nonnormal}
EXPM_SCALES = [-0.05j, -3j, -100j, -3000j, -0.7, -20.0, 5.0, 0.3 - 2j]
EXPM_MAX = 1e250    # real scales whose exponential would exceed this are left out


# ---------------------------------------------------------------------------------------------------------------------
# B. the reference-Lanczos exact-basis tridiagonal
def lanczos_ref_tridiag(n, im_a0=0.0, seed=0):
    """diag (a0, b0, 0, ..., 0), off-diagonals b_l in [0.2, 1.5), scaled to |Re T|_1 = 1; Im a0 is set after scaling."""
    rng = np.random.default_rng(3000 + 17 * n + seed)
    b = rng.uniform(0.2, 1.5, n - 1)
    T = np.diag(b, 1) + np.diag(b, -1)
    T[0, 0] = 0.3
    if n > 1:
        T[1, 1] = b[0]
    T = T / norm1(T)
    T = T.astype(np.complex128)
    T[0, 0] += 1j * im_a0
    return T


# ---------------------------------------------------------------------------------------------------------------------
# emulation of the recurrences on the unit-vector inputs (premise checks on the CPU)
def arnoldi_basis(H):
    """One-pass classical Gram-Schmidt Arnoldi on H from e_0, as the kernels order it; returns (V, beta)."""
    n = H.shape[0]
    V, betas = [e0(n)], []
    for l in range(n):  # noqa: E741
        w = H @ V[-1]
        Vm = np.array(V)
        h = np.conj(Vm) @ w
        w = w - h @ Vm
        b = float(np.sqrt(np.sum(w.real ** 2 + w.imag ** 2)))
        betas.append(b)
        if b > 1e-12:
            V.append(rdiv(w, b))
        else:
            break
    return np.array(V), np.array(betas)


def lanczos_ref_basis(T):
    """The reference recurrence alpha_l = <v_0|T v_l>; returns (V, alpha, beta)."""
    n = T.shape[0]
    v0 = e0(n)
    V, alphas, betas = [v0], [], []
    for l in range(n):  # noqa: E741
        w = T @ V[-1]
        a = np.vdot(v0, w)
        alphas.append(a)
        w = w - a * V[-1] - (betas[-1] * V[-2] if l > 0 else 0)
        b = float(np.sqrt(np.sum(w.real ** 2 + w.imag ** 2)))
        betas.append(b)
        if b < 1e-12:
            break
        V.append(rdiv(w, b))
    return np.array(V), np.array(alphas), np.array(betas)


def textbook_lanczos_basis(a, b):
    """Textbook Lanczos (alpha_i = Re <v_i|T v_i>) on the real symmetric tridiagonal (a, b) from e_0."""
    n = len(a)
    T = np.diag(a) + np.diag(b, 1) + np.diag(b, -1)
    V, alphas, betas = [e0(n)], [], []
    for i in range(n):
        w = T @ V[-1]
        al = np.vdot(V[-1], w).real
        alphas.append(al)
        w = w - al * V[-1] - (betas[-1] * V[-2] if i > 0 else 0)
        bb = float(np.sqrt(np.sum(w.real ** 2 + w.imag ** 2)))
        betas.append(bb)
        if bb < 1e-12:
            break
        V.append(rdiv(w, bb))
    return np.array(V), np.array(alphas), np.array(betas)


# ---------------------------------------------------------------------------------------------------------------------
# G. real symmetric tridiagonals for the Lanczos eigensolver
def wilkinson21():
    return np.abs(np.arange(-10, 11)).astype(float), np.ones(20)


def tridiag_family(name, n, seed=0):
    """(a, b) of an n x n real symmetric tridiagonal with nonzero off-diagonals."""
    rng = np.random.default_rng(4000 + 31 * n + seed)
    if name == "random":
        return rng.standard_normal(n), rng.uniform(0.1, 2.0, n - 1)
    if name == "laplacian-":
        return np.full(n, 2.0), np.full(n - 1, -1.0)
    if name == "laplacian+":
        return np.full(n, 2.0), np.full(n - 1, 1.0)
    if name == "graded":      # entries from 1 down to 1e-8
        g = np.logspace(0, -8, n)
        return g * rng.standard_normal(n), g[:-1] * rng.uniform(0.5, 1.0, n - 1)
    if name == "negdef":      # T - (|T| + 1) I: every eigenvalue below -1
        a, b = rng.standard_normal(n), rng.uniform(0.1, 2.0, n - 1)
        return a - (np.abs(a).max() + 2 * 2.0 + 1.0), b
    if name in ("scaled1e6", "scaled1e-6"):
        s = 1e6 if name == "scaled1e6" else 1e-6
        return s * rng.standard_normal(n), s * rng.uniform(0.1, 2.0, n - 1)
    raise ValueError(name)


def tridiag_dense(a, b):
    return np.diag(a) + np.diag(b, 1) + np.diag(b, -1)


def _sturm_count(a, b, x):
    """Number of eigenvalues < x of the symmetric tridiagonal (a, b) (mpmath numbers)."""
    cnt = 0
    q = a[0] - x
    tiny = mpmath.mpf(10) ** (-2 * mpmath.mp.dps)
    if q < 0:
        cnt += 1
    for i in range(1, len(a)):
        if q == 0:
            q = tiny
        q = a[i] - x - b[i - 1] ** 2 / q
        if q < 0:
            cnt += 1
    return cnt


@functools.lru_cache(maxsize=None)
def _mp_extreme_eigenvalue(abuf, bbuf, root, dps):
    a64 = np.frombuffer(abuf, dtype=np.float64)
    b64 = np.frombuffer(bbuf, dtype=np.float64)
    n = len(a64)
    with mpmath.workdps(dps):
        a = [mpmath.mpf(float(x)) for x in a64]
        b = [mpmath.mpf(float(x)) for x in b64]
        r = [(abs(b[i - 1]) if i > 0 else 0) + (abs(b[i]) if i < n - 1 else 0) for i in range(n)]
        lo = min(a[i] - r[i] for i in range(n)) - 1
        hi = max(a[i] + r[i] for i in range(n)) + 1
        target = 1 if root == 0 else n          # smallest lambda with count(< lambda) >= target
        width = hi - lo
        while hi - lo > width * mpmath.mpf(10) ** (-dps + 5):
            mid = (lo + hi) / 2
            if _sturm_count(a, b, mid) >= target:
                hi = mid
            else:
                lo = mid
        return float((lo + hi) / 2)


def mp_extreme_eigenvalue(a, b, root):
    """The smallest (root 0) or largest eigenvalue of the tridiagonal (a, b) by Sturm bisection at 40 digits."""
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    return _mp_extreme_eigenvalue(a.tobytes(), b.tobytes(), int(root != 0), EIG_DPS)


def tridiag_reference(a, b, root):
    """(lambda, v, gap, |T|): the extreme eigenvalue at 40 digits, its eigenvector from LAPACK (eigh_tridiagonal: the
    angle bar 64 n EPS |T| / gap needs only a backward-stable vector) and the distance to the next eigenvalue."""
    n = len(a)
    lam = mp_extreme_eigenvalue(a, b, root)
    if n == 1:
        return lam, np.ones(1), np.inf, abs(a[0])
    w, V = scipy.linalg.eigh_tridiagonal(a, b)
    i = 0 if root == 0 else n - 1
    gap = abs(w[1] - w[0]) if root == 0 else abs(w[-1] - w[-2])
    nT = float(np.abs(w).max())
    return lam, V[:, i], gap, nT


# ---------------------------------------------------------------------------------------------------------------------
# D. Kronecker operators with a k-dimensional invariant subspace
def _unitary(rng, n):
    Q, R = np.linalg.qr(crand(rng, n, n))
    return Q * (np.diag(R) / np.abs(np.diag(R)))[None, :]


def invariant_factor(rng, n, k):
    """F = Q blkdiag(A, B) Q^H with non-Hermitian A (k x k), B; returns (F, Q[:, :k], A).  The eigenvalues of A are
    spread over an annulus so that the Krylov space of a generic start vector fills range(Q[:, :k]); |B| ~ 0.1 keeps the
    rest of the spectrum inside that annulus."""
    Q = _unitary(rng, n)
    ang = rng.uniform(0, 2 * np.pi, k) if k > 1 else np.zeros(1)
    lam = (0.5 + 0.5 * np.arange(k) / max(k - 1, 1)) * np.exp(1j * (ang + 2 * np.pi * np.arange(k) / max(k, 1)))
    X = np.eye(k) + 0.3 * crand(rng, k, k)
    A = X @ np.diag(lam) @ np.linalg.inv(X)
    B = 0.05 * crand(rng, n - k, n - k) / np.sqrt(max(n - k, 1))    # small: rounding outside the subspace is not amplified
    M = np.zeros((n, n), dtype=np.complex128)
    M[:k, :k] = A
    M[k:, k:] = B
    return Q @ M @ Q.conj().T, Q[:, :k], A


def kron_breakdown_case(dims, ks, seed=4):
    """H = L (x) W (x) R (dense factors of sizes ``dims``) with psi in the product of k_f-dimensional invariant
    subspaces, so the Krylov space of psi has dimension prod(ks).  Returns (Lm, Wm, Rm, psi, P, Ak, c): psi = P c with the
    orthonormal P (N x k), and H P = P Ak."""
    rng = np.random.default_rng(5000 + seed + 7 * sum(dims) + 131 * int(np.prod(ks)))
    facs = [invariant_factor(rng, n, k) for n, k in zip(dims, ks, strict=True)]
    cs = []
    for _, _, A in facs:
        c = crand(rng, A.shape[0])
        cs.append(c / np.linalg.norm(c))
    P = np.kron(np.kron(facs[0][1], facs[1][1]), facs[2][1])
    Ak = np.kron(np.kron(facs[0][2], facs[1][2]), facs[2][2])
    c = np.kron(np.kron(cs[0], cs[1]), cs[2])
    psi = (P @ c).reshape(dims)
    return facs[0][0], facs[1][0], facs[2][0], psi, P, Ak, c


def kron_matvec(Lm, Wm, Rm):
    """H psi for H = Lm (x) Wm (x) Rm on psi of shape (Dl, d, Dr): what heff_term computes for L = Lm[:, None, :],
    W = Wm[None, :, :, None] and R = Rm[:, None, :]."""
    return lambda v: np.einsum("ab,ij,rs,bjs->air", Lm, Wm, Rm, v, optimize=True)
