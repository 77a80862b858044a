"""CPU oracle for the TDVP hot path -- TEST INFRASTRUCTURE, NOT A PRODUCT PATH.

A plain NumPy/SciPy restatement of what PyTDSCF 1.3.3 (reference at /root/reference) does on its
MPS/MPO one-site projector-splitting TDVP path.  Only ``tests/``, ``__graft_entry__.smoke()`` and
``bench.py``'s cpu_baseline / ``--impl reference`` arm may import this module; the product
(``pytdscf_b200``) never does and has no CPU fallback.

Parity pin: every public function here is checked against the UNMODIFIED reference run in the build
container under ``oracle/refshim`` (``tests/golden/make_golden.py`` -> ``tests/golden/*.npz``,
``tests/test_oracle_golden.py``).  Third-party arithmetic that the reference delegates to
``opt_einsum`` 3.4.0 (pairwise contraction order) and LAPACK is restated with ``np.einsum`` on an
unlimited-memory greedy path and ``scipy.linalg`` -- summation order inside those is unpinned in the
reference itself (SURVEY F7).

Scope: ``nstate == 1`` (every MPO configuration of the reference uses one "state" with electronic
levels as an exciton site), standard method (no SPF layer), time-independent Hamiltonian.

Reference map (file:line relative to /root/reference):
  MPOHamiltonian / SiteCore        pytdscf/_mpo_cls.py:44-234
  env_update_term                  pytdscf/_contraction.py:148-397   (contract_with_site_mpo)
  heff_term / heff_apply           pytdscf/_contraction.py:1038-1243 (multiplyH_MPS_direct_MPO)
  keff_term / keff_apply           pytdscf/_contraction.py:1297-1407 (multiplyK_MPS_direct_MPO)
  sil_reference                    pytdscf/_integrator.py:453-655    (short_iterative_lanczos)
  sia_reference                    pytdscf/_integrator.py:287-432    (short_iterative_arnoldi)
  lanczos_ground_state             pytdscf/_integrator.py:74-138     (matrix_diagonalize_lanczos)
  shift_qr / shift_lq              pytdscf/_site_cls.py:138-292      (SiteCoef.gauge_trf)
  truncate_bond                    pytdscf/_site_cls.py:586-690      (truncate_sigvec)
  bond_dims / initial_mps          pytdscf/_mps_cls.py:2616-2703 ; pytdscf/_site_cls.py:409-476
  zero_site_block / renormalize    pytdscf/_mps_mpo.py:364-419, 421-696
  terms_for_heff / terms_for_keff  pytdscf/_mps_mpo.py:698-858, 860-1021
  TDVPOracle.sweep / propagate     pytdscf/_mps_cls.py:798-1014, 452-503, 1016-1206, 1739-1850
  TDVPOracle.energy / autocorr     pytdscf/_mps_cls.py:540-612 ; pytdscf/wavefunction.py:226-257
"""
from __future__ import annotations

import cmath
import math
from dataclasses import dataclass, field

import numpy as np
import scipy.linalg

EPS_KRYLOV = 1e-12  # _integrator.py:22
KRYLOV_CAP = 20  # _integrator.py:182
SQRT_EPSRHO = 1e-4  # _site_cls.py:22

# --------------------------------------------------------------------------------------
# einsum helper: pairwise BLAS-backed contraction on an unlimited-memory greedy path
# (what opt_einsum.contract does by default; np.einsum(optimize=True) must NOT be used, SURVEY F6)
# --------------------------------------------------------------------------------------
_PATHS: dict = {}


def _einsum(sub: str, *ops: np.ndarray) -> np.ndarray:
    key = (sub,) + tuple(o.shape for o in ops)
    path = _PATHS.get(key)
    if path is None:
        path = np.einsum_path(sub, *ops, optimize=("greedy", 2**62))[0]
        _PATHS[key] = path
    return np.einsum(sub, *ops, optimize=path)


# --------------------------------------------------------------------------------------
# MPO container
# --------------------------------------------------------------------------------------
@dataclass
class SiteCore:
    """One MPO core acting at ``psite`` (``_mpo_cls.py:166-199``).

    ``data`` is ``None`` for an identity gap core (reference: ``data=1``), a 3-index array
    (w_l, d, w_r) for a diagonal core, or a 4-index array (w_l, d_bra, d_ket, w_r)."""

    key: tuple
    psite: int
    data: np.ndarray | None
    is_left: bool
    is_right: bool

    @property
    def diag(self) -> bool:
        return self.data is None or self.data.ndim == 3


class MPOHamiltonian:
    """``{key: [cores]}`` -> per-site core lists (``_mpo_cls.py:116-163``), plus the scalar ``coupleJ``."""

    def __init__(self, nsite: int, operators: dict, coupleJ: complex = 0.0):
        self.nsite = nsite
        self.coupleJ = coupleJ
        self.operators = operators
        self.calc_point: list[list[SiteCore]] = [[] for _ in range(nsite)]
        for key, cores in operators.items():
            sites = []
            for ind, core in zip(key, cores, strict=True):
                if isinstance(ind, tuple):
                    if len(ind) != core.ndim - 2 or len(set(ind)) != 1:
                        raise ValueError(f"bad MPO key entry {ind} for core of shape {core.shape}")
                    sites.append(ind[0])
                else:
                    if core.ndim != 3:
                        raise ValueError(f"bad MPO key entry {ind} for core of shape {core.shape}")
                    sites.append(int(ind))
            lo, hi = min(sites), max(sites)
            for s, core in zip(sites, cores, strict=True):
                self.calc_point[s].append(SiteCore(key, s, np.asarray(core), s == lo, s == hi))
            for s in range(lo + 1, hi):
                if s not in sites:
                    self.calc_point[s].append(SiteCore(key, s, None, False, False))


# --------------------------------------------------------------------------------------
# contractions
# --------------------------------------------------------------------------------------
def env_update_term(gauge: str, bra: np.ndarray, ket: np.ndarray, E, core) -> np.ndarray:
    """New environment block from site tensors, old block ``E`` and a core.

    ``E``: ``None`` (identity) or (D, w, D) array; ``core``: ``None``/gap (identity), or SiteCore.
    ``bra`` is conjugated here.  Result always has 3 indices (``_contraction.py:395-396``)."""
    cb = np.conj(bra)
    W = None if core is None else core.data
    if gauge == "A":
        if W is None and E is None:
            out = _einsum("nsi,nsj->ij", cb, ket)
        elif W is None:
            out = _einsum("msi,nsj,mpn->ipj", cb, ket, E)
        elif E is None:
            assert W.shape[0] == 1
            if W.ndim == 3:
                out = _einsum("mri,mrj,rq->iqj", cb, ket, W[0])
            else:
                out = _einsum("mri,msj,rsq->iqj", cb, ket, W[0])
        elif W.ndim == 3:
            out = _einsum("mri,nrj,mpn,prq->iqj", cb, ket, E, W)
        else:
            out = _einsum("mri,nsj,mpn,prsq->iqj", cb, ket, E, W)
    elif gauge == "B":
        if W is None and E is None:
            out = _einsum("isn,jsn->ij", cb, ket)
        elif W is None:
            out = _einsum("ism,jsn,mqn->iqj", cb, ket, E)
        elif E is None:
            assert W.shape[-1] == 1
            if W.ndim == 3:
                out = _einsum("irm,jrm,pr->ipj", cb, ket, W[:, :, 0])
            else:
                out = _einsum("irm,jsm,prs->ipj", cb, ket, W[:, :, :, 0])
        elif W.ndim == 3:
            out = _einsum("irm,jrn,mqn,prq->ipj", cb, ket, E, W)
        else:
            out = _einsum("irm,jsn,mqn,prsq->ipj", cb, ket, E, W)
    else:
        raise ValueError(gauge)
    if out.ndim == 2:
        out = out[:, None, :]
    return out


def heff_term(L, core, R, psi: np.ndarray) -> np.ndarray:
    """One MPO term of H_eff.psi (``_contraction.py:1089-1161``; 3-index/identity operands only).

    NB the identity-core case with 3-index L and R sums the two MPO bonds independently
    ("bjs,acb,rts->ajr"), exactly as the reference does."""
    W = None if core is None else core.data
    ops = [psi]
    lhs = ["bjs"]
    a, i, r = "b", "j", "s"
    if L is not None:
        ops.append(L)
        lhs.append("acb")
        a = "a"
    if W is not None:
        ops.append(W)
        if W.ndim == 3:
            lhs.append("cjt")
        else:
            lhs.append("cijt")
            i = "i"
    if R is not None:
        ops.append(R)
        lhs.append("rts")
        r = "r"
    if len(ops) == 1:
        return psi
    return _einsum(",".join(lhs) + "->" + a + i + r, *ops)


def keff_term(L, R, sigma: np.ndarray) -> np.ndarray:
    """One term of K_eff.sigma (``_contraction.py:1314-1339``)."""
    if L is None and R is None:
        return sigma
    if L is None:
        return _einsum("as,rcs->ar", sigma, R)
    if R is None:
        return _einsum("br,acb->ar", sigma, L)
    return _einsum("bs,acb,rcs->ar", sigma, L, R)


def heff_apply(terms: dict, coupleJ, psi: np.ndarray) -> np.ndarray:
    """Sum over terms in the reference's order (``_contraction.py:1182-1243``)."""
    out = None
    if coupleJ != 0.0:
        out = heff_term(*terms["ovlp"], psi) * coupleJ
    for key, (L, core, R) in terms.items():
        if key == "ovlp":
            continue
        add = heff_term(L, core, R, psi)
        if out is None:
            out = add if add is not psi else psi.copy()
        else:
            out += add
    return out


def keff_apply(terms: dict, coupleJ, sigma: np.ndarray) -> np.ndarray:
    out = None
    if coupleJ != 0.0:
        out = keff_term(*terms["ovlp"], sigma) * coupleJ
    for key, (L, R) in terms.items():
        if key == "ovlp":
            continue
        add = keff_term(L, R, sigma)
        if out is None:
            out = add if add is not sigma else sigma.copy()
        else:
            out += add
    return out


# --------------------------------------------------------------------------------------
# Krylov exponentials, exactly as the reference runs them (SURVEY Appendix B)
# --------------------------------------------------------------------------------------
def krylov_warmup(maxsize: int, last_niter: int) -> tuple[int, int]:
    """(ndim, n_warmup) of ``_integrator.py:178-186``."""
    ndim = min(maxsize, KRYLOV_CAP)
    n_warm = min(maxsize, min(max(0, last_niter - 2), 15))
    return ndim, n_warm


def _rescale(y, b0, conserve_norm):
    if conserve_norm:
        return y / float(np.linalg.norm(y))
    return y * b0


def sil_reference(scale, matvec, psi, thresh, *, last_niter=0, conserve_norm=True, maxsize=None, small_expm=None):
    """exp(scale*H) psi by the reference's three-term recurrence (alpha_l = <v0|H v_l>).

    ``matvec`` maps an array of ``psi.shape`` to one of the same shape.  Returns (psi_new, niter).
    ``small_expm``: optional callable A -> expm(A)[:, 0] for the k x k matrix A = scale * T (k >= 2) that replaces the
    reference's eigh_tridiagonal / eig step, e.g. a high-precision exponential; None keeps the reference's arithmetic."""
    shape = psi.shape
    maxsize = psi.size if maxsize is None else int(maxsize)   # adaptive runs: size of the tensor before it was extended
    ndim, n_warm = krylov_warmup(maxsize, last_niter)
    v0 = psi.reshape(-1).astype(np.complex128, copy=True)
    if conserve_norm:
        b0 = 1.0
    else:
        b0 = float(np.linalg.norm(v0))
        if b0 == 0.0:
            raise ValueError("Initial psi has zero norm.")
        v0 /= b0
    v0c = np.conj(v0)
    V = [v0]
    alpha: list[complex] = []
    beta: list[float] = []
    alpha_is_real = True
    prev = None
    for l in range(ndim):  # noqa: E741
        w = matvec(psi if l == 0 else V[-1].reshape(shape)).reshape(-1)
        if w is psi or np.shares_memory(w, psi):
            w = w.copy()
        if not conserve_norm and l == 0:
            w /= b0
        a = complex(np.inner(v0c, w))
        alpha.append(a)
        w -= V[-1] * a
        if l > 0:
            w -= V[-2] * beta[-1]
        b = float(scipy.linalg.norm(w))
        beta.append(b)
        if b >= EPS_KRYLOV:
            w /= b
        V.append(w)
        conv = b < EPS_KRYLOV or l + 1 == maxsize
        if alpha_is_real and abs(a.imag) > 1e-10:
            alpha_is_real = False
        if l < n_warm and not conv:
            continue
        if l == 0:
            y = v0 * cmath.exp(scale * alpha[0])
        elif small_expm is not None:
            T = (
                np.diag(np.real(alpha) if alpha_is_real else np.asarray(alpha), 0).astype(np.complex128)
                + np.diag(beta[:-1], -1)
                + np.diag(beta[:-1], 1)
            )
            y = np.dot(small_expm(scale * T), np.asarray(V[:-1]))
        else:
            if alpha_is_real:
                lam, phi = scipy.linalg.eigh_tridiagonal(np.real(alpha), beta[:-1])
                c = phi @ (np.exp(scale * lam) * np.conjugate(phi).T[:, 0])
            else:
                T = (
                    np.diag(alpha, 0)
                    + np.diag(beta[:-1], -1).astype(np.complex128)
                    + np.diag(beta[:-1], 1).astype(np.complex128)
                )
                lam, phi = scipy.linalg.eig(T)
                e0 = np.zeros(l + 1, dtype=T.dtype)
                e0[0] = 1
                c = phi @ (np.exp(scale * lam) * np.linalg.solve(phi, e0))
            y = np.dot(c, np.asarray(V[:-1]))
        if conv:
            return _rescale(y, b0, conserve_norm).reshape(shape), l + 1
        if prev is not None and float(np.linalg.norm(y - prev)) < thresh:
            return _rescale(y, b0, conserve_norm).reshape(shape), l + 1
        prev = y
    raise ValueError("Short Iterative Lanczos is not converged")


def sia_reference(scale, matvec, psi, thresh, *, last_niter=0, conserve_norm=True, maxsize=None, small_expm=None):
    """Arnoldi variant: one-pass classical Gram-Schmidt, dense eig of the Hessenberg block (``small_expm`` as in
    ``sil_reference``, applied to scale times the Hessenberg block)."""
    shape = psi.shape
    maxsize = psi.size if maxsize is None else int(maxsize)
    ndim, n_warm = krylov_warmup(maxsize, last_niter)
    hess = np.zeros((ndim + 1, ndim), dtype=np.complex128)
    v0 = psi.reshape(-1).astype(np.complex128, copy=True)
    if conserve_norm:
        b0 = 1.0
    else:
        b0 = float(np.linalg.norm(v0))
        if b0 == 0.0:
            raise ValueError("Initial psi has zero norm.")
        v0 /= b0
    V = v0[None, :].copy()
    v = v0
    prev = None
    for l in range(ndim):  # noqa: E741
        w = matvec(psi if l == 0 else v.reshape(shape)).reshape(-1)
        if np.shares_memory(w, psi):
            w = w.copy()
        if not conserve_norm and l == 0:
            w /= b0
        h = np.sum(np.conj(V) * w[None, :], axis=1)
        w -= np.sum(h[:, None] * V, axis=0)
        b = float(np.linalg.norm(w))
        hess[: l + 1, l] = h
        if b > EPS_KRYLOV:
            w /= b
            V = np.vstack([V, w])
            if hess.shape[0] > l + 1:
                hess[l + 1, l] = b
        v = w
        conv = b < EPS_KRYLOV or l + 1 == maxsize
        if l < n_warm and not conv:
            continue
        if l == 0:
            y = v0 * cmath.exp(scale * hess[0, 0])
        elif small_expm is not None:
            c = small_expm(scale * hess[: l + 1, : l + 1])
            y = np.tensordot(c, V[: c.shape[0], :], axes=(0, 0))
        else:
            sub = hess[: l + 1, : l + 1]
            lam, phi = np.linalg.eig(sub)
            e0 = np.zeros(l + 1, dtype=sub.dtype)
            e0[0] = 1
            c = phi @ (np.exp(scale * lam) * np.linalg.solve(phi, e0))
            y = np.tensordot(c, V[: c.shape[0], :], axes=(0, 0))
        if conv:
            return _rescale(y, b0, conserve_norm).reshape(shape), l + 1
        if prev is not None and float(np.linalg.norm(y - prev)) < thresh:
            return _rescale(y, b0, conserve_norm).reshape(shape), l + 1
        prev = y
    raise ValueError("Short Iterative Arnoldi is not converged in 20 basis")


def lanczos_ground_state(matvec, psi, root=0, thresh=1e-9):
    """Textbook Lanczos eigen-solver of the improved-relaxation path. Returns (vec, niter)."""
    shape = psi.shape
    ndim = psi.size
    n_iter = min(ndim, 3000)
    alpha: list[float] = []
    beta: list[float] = [0.0]
    vecs = [psi.reshape(-1).astype(np.complex128, copy=True)]
    prev = None
    for it in range(n_iter + 1):
        w = matvec(vecs[-1].reshape(shape)).reshape(-1).copy()
        alpha.append(float(np.inner(np.conj(vecs[-1]), w).real))
        w -= vecs[-1] * alpha[-1]
        if len(vecs) >= 2:
            w -= vecs[-2] * beta[-1]
        beta.append(float(scipy.linalg.norm(w)))
        w /= beta[-1]
        _, phi = scipy.linalg.eigh_tridiagonal(np.array(alpha), np.array(beta[1:-1]))
        y = np.asarray(vecs).T @ phi[:, root]
        if abs(beta[-1]) < EPS_KRYLOV:
            return y.reshape(shape), it + 1
        if it > 0:
            if float(scipy.linalg.norm(y - prev)) < thresh or it == ndim:
                return y.reshape(shape), it + 1
        prev = y
        vecs.append(w)
    raise ValueError("Lanczos Diagonalization is not converged in 3000 basis")


# --------------------------------------------------------------------------------------
# gauge shifts
# --------------------------------------------------------------------------------------
def _regularize(psi: np.ndarray) -> np.ndarray:
    dl, d, dr = psi.shape
    U, s, Vh = scipy.linalg.svd(np.ascontiguousarray(psi.transpose(0, 2, 1).reshape(-1, d)), full_matrices=False)
    s = np.where(s > SQRT_EPSRHO, s, s + SQRT_EPSRHO * np.exp(-s / SQRT_EPSRHO))
    return (U @ (np.diag(s) @ Vh)).reshape(dl, dr, d).transpose(0, 2, 1)


def shift_qr(psi: np.ndarray, regularize: bool = False):
    """Psi(Dl,d,Dr) -> A(Dl,d,k), sigma(k,Dr): economic Householder QR of the (Dl*d) x Dr matrix."""
    if regularize:
        psi = _regularize(psi)
    dl, d, dr = psi.shape
    Q, R = scipy.linalg.qr(psi.reshape(dl * d, dr), mode="economic")
    return Q.reshape(dl, d, -1), R


def shift_lq(psi: np.ndarray, regularize: bool = False):
    """Psi(Dl,d,Dr) -> sigma(Dl,k), B(k,d,Dr): QR of the transposed (Dr*d) x Dl matrix."""
    if regularize:
        psi = _regularize(psi)
    dl, d, dr = psi.shape
    Q, R = scipy.linalg.qr(np.ascontiguousarray(psi.transpose(2, 1, 0).reshape(dr * d, dl)), mode="economic")
    return R.T, Q.reshape(dr, d, -1).transpose(2, 1, 0)


def truncate_bond(A, sigma, B, p, regularize=False, keepdim=False):
    """SVD of the bond matrix, cumulative singular-VALUE weight truncation (``_site_cls.py:620-690``).

    ``A``/``B`` may be ``None``.  Returns (A.U or U, diag(s/|s|), Vh.B or Vh, rank)."""
    U, s, Vh = scipy.linalg.svd(sigma, full_matrices=False)
    csum = np.cumsum(s.real)
    idx = int(np.argmax(csum / csum[-1] >= (1 - p)) + 1)
    s_thin = s[:idx]
    if not keepdim:
        U = U[:, :idx]
        Vh = Vh[:idx, :]
    Lout = U if A is None else np.tensordot(A, U, axes=(2, 0))
    Rout = Vh if B is None else np.tensordot(Vh, B, axes=(1, 0))
    if regularize and sigma.shape != (1, 1):
        s_thin = np.where(s_thin > SQRT_EPSRHO, s_thin, s_thin + SQRT_EPSRHO * np.exp(-s_thin / SQRT_EPSRHO))
    nrm = np.linalg.norm(s_thin)
    if keepdim:
        full = np.zeros_like(s)
        full[:idx] = s_thin
        new_sigma = np.diag(full / nrm)
    else:
        new_sigma = np.diag(s_thin / nrm)
    return Lout, new_sigma, Rout, idx


# --------------------------------------------------------------------------------------
# initial MPS
# --------------------------------------------------------------------------------------
def bond_dims(dims: list[int], isite: int, m: int) -> tuple[int, int]:
    n = len(dims)
    dim_left = 1 if isite == 0 else min(m, math.prod(dims[:isite]))
    dim_right = 1 if isite == n - 1 else min(m, math.prod(dims[isite + 1 :]))
    dc = dims[isite]
    return min(dim_left, dc * dim_right, m), min(dim_left * dc, dim_right, m)


def initial_mps(dims, m, core_weights, *, space="hilbert", scale=1.0):
    """Zero-padded Hartree product, right-canonicalised by LQ sweeps; site 0 is the centre ("Psi").

    ``core_weights[i]`` is a 1-D weight vector (normalised per site: 2-norm in Hilbert space, trace of the
    reshaped sqrt(d) x sqrt(d) matrix in Liouville space) or a 3-D core copied into the top-left corner."""
    n = len(dims)
    cores = []
    for i in range(n):
        ml, mr = bond_dims(dims, i, m)
        data = np.zeros((1 if i == 0 else ml, dims[i], 1 if i == n - 1 else mr), dtype=np.complex128)
        w = np.array(core_weights[i], dtype=np.complex128)
        if w.ndim == 1:
            data[0, :, 0] = w
            if space == "hilbert":
                data[0, :, 0] /= np.linalg.norm(w)
            else:
                q = math.isqrt(dims[i])
                data[0, :, 0] /= np.trace(w.reshape(q, q))
        elif w.ndim == 3:
            a, b, c = w.shape
            data[:a, :b, :c] = w
        else:
            raise ValueError("core weight must be 1-D or 3-D")
        cores.append(data)
    for i in range(n - 1, 0, -1):
        sig, B = shift_lq(cores[i])
        cores[i] = B
        cores[i - 1] = np.tensordot(cores[i - 1], sig, axes=(2, 0))
    if space == "hilbert":
        cores[0] = cores[0] * (scale / np.linalg.norm(cores[0]))
    else:
        cores[0] = cores[0] * scale
    return cores


# --------------------------------------------------------------------------------------
# environment bookkeeping
# --------------------------------------------------------------------------------------
@dataclass
class Block:
    data: np.ndarray
    is_identity: bool = False


def zero_site_block() -> dict:
    return {"ovlp": Block(np.ones((1, 1, 1), dtype=complex), True)}


def renormalize(psite: int, site: np.ndarray, gauge: str, blocks: dict, H: MPOHamiltonian, A_is_sys: bool) -> dict:
    """Absorb site ``psite`` (bra == ket) into the system blocks."""
    nxt: dict = {}
    ov = blocks["ovlp"]
    if ov.is_identity:
        dim = site.shape[2] if gauge == "A" else site.shape[0]
        nxt["ovlp"] = Block(np.eye(dim, dtype=complex)[:, None, :], True)
        E_ovlp = None
    else:
        nxt["ovlp"] = Block(env_update_term(gauge, site, site, ov.data, None), False)
        E_ovlp = ov.data
    for core in H.calc_point[psite]:
        if (core.is_left and A_is_sys) or (core.is_right and not A_is_sys):
            E = E_ovlp
        else:
            E = blocks[core.key]
        new = env_update_term(gauge, site, site, E, core)
        if (core.is_right and A_is_sys) or (core.is_left and not A_is_sys):
            if "summed" in nxt:
                nxt["summed"] += new
            else:
                nxt["summed"] = new
        else:
            nxt[core.key] = new
    if "summed" in blocks:
        new = env_update_term(gauge, site, site, blocks["summed"], None)
        if "summed" in nxt:
            nxt["summed"] += new
        else:
            nxt["summed"] = new
    return nxt


def _ovlp_operand(blocks):
    ov = blocks["ovlp"]
    return None if ov.is_identity else ov.data


def terms_for_heff(psite, op_sys, op_env, H: MPOHamiltonian, A_is_sys: bool) -> dict:
    Lb, Rb = (op_sys, op_env) if A_is_sys else (op_env, op_sys)
    Lo, Ro = _ovlp_operand(Lb), _ovlp_operand(Rb)
    terms = {"ovlp": (Lo, None, Ro)}
    if "summed" in Lb:
        terms["summ_l"] = (Lb["summed"], None, Ro)
    if "summed" in Rb:
        terms["summ_r"] = (Lo, None, Rb["summed"])
    for core in H.calc_point[psite]:
        terms[core.key] = (Lb.get(core.key, Lo), core, Rb.get(core.key, Ro))
    return terms


def terms_for_keff(op_sys, op_env, A_is_sys: bool) -> dict:
    Lb, Rb = (op_sys, op_env) if A_is_sys else (op_env, op_sys)
    Lo, Ro = _ovlp_operand(Lb), _ovlp_operand(Rb)
    terms = {"ovlp": (Lo, Ro)}
    if "summed" in Lb:
        terms["summ_l"] = (Lb["summed"], Ro)
    if "summed" in Rb:
        terms["summ_r"] = (Lo, Rb["summed"])
    for key in op_sys.keys():
        if key in ("summed", "ovlp"):
            continue
        terms[key] = (Lb[key], Rb[key])
    return terms


# --------------------------------------------------------------------------------------
# the sweep driver
# --------------------------------------------------------------------------------------
@dataclass
class TDVPOracle:
    """One-site projector-splitting TDVP of an MPS under an MPO Hamiltonian (serial reference path)."""

    H: MPOHamiltonian
    mps: list  # list of (Dl, d, Dr) complex128 arrays; site 0 is the orthogonality centre
    thresh: float = 1e-9
    integrator: str = "lanczos"
    conserve_norm: bool = True
    space: str = "hilbert"
    relax: bool | str = False
    gauges: list = field(default_factory=list)
    niter: dict = field(default_factory=dict)  # shared per-site Krylov history (SURVEY F3)
    trace: list = field(default_factory=list)  # [("H"|"K", site, niter)]
    op_sys_sites: list | None = None

    def __post_init__(self):
        if not self.gauges:
            self.gauges = ["Psi"] + ["B"] * (len(self.mps) - 1)
        if self.space == "liouville":
            self.conserve_norm = False

    # -- environments ---------------------------------------------------------------
    def build_envs(self, begin: int, end: int, H: MPOHamiltonian | None = None) -> list:
        """Blocks obtained by absorbing sites begin, begin+-1, ... (excluding ``end``)."""
        H = self.H if H is None else H
        left = begin < end
        step = 1 if left else -1
        blocks = [zero_site_block()]
        for p in range(begin, end, step):
            blocks.append(renormalize(p, self.mps[p], "A" if left else "B", blocks[-1], H, left))
        return blocks

    # -- local exponentials ---------------------------------------------------------
    def _expm(self, scale_sign: complex, dt: float, matvec, x, site: int, kind: str):
        last = self.niter.get(site, 0)
        if self.relax == "improved":
            if kind == "K":
                return x
            y, n = lanczos_ground_state(matvec, x)
            y = y / np.linalg.norm(y)
        else:
            if self.relax:
                scale = (scale_sign * -1j).real * (dt / 2)  # imaginary time: -dt/2 for H, +dt/2 for K
            else:
                scale = scale_sign * (dt / 2)
            solver = sia_reference if (self.integrator == "arnoldi" and not self.relax) else sil_reference
            y, n = solver(scale, matvec, x, self.thresh, last_niter=last, conserve_norm=self.conserve_norm)
            if self.relax and self.conserve_norm:
                y = y / np.linalg.norm(y)
        self.niter[site] = n
        self.trace.append((kind, site, n))
        return y

    # -- one half sweep -------------------------------------------------------------
    def sweep(self, dt: float, begin: int, end: int):
        A_is_sys = begin <= end
        step = 1 if A_is_sys else -1
        H = self.H
        op_sys = zero_site_block()
        if self.op_sys_sites is None:
            env_sites = self.build_envs(end, begin)
        else:
            env_sites = self.op_sys_sites[:]
        self.op_sys_sites = [op_sys]
        for p in range(begin, end + step, step):
            op_env = env_sites.pop()
            terms = terms_for_heff(p, op_sys, op_env, H, A_is_sys)
            self.mps[p] = self._expm(-1.0j, dt, lambda x, t=terms: heff_apply(t, H.coupleJ, x), self.mps[p], p, "H")
            self.gauges[p] = "Psi"
            if p == end:
                break
            if A_is_sys:
                self.mps[p], sigma = shift_qr(self.mps[p])
                self.gauges[p] = "A"
            else:
                sigma, self.mps[p] = shift_lq(self.mps[p])
                self.gauges[p] = "B"
            op_sys = renormalize(p, self.mps[p], self.gauges[p], op_sys, H, A_is_sys)
            kterms = terms_for_keff(op_sys, op_env, A_is_sys)
            sigma = self._expm(+1.0j, dt, lambda x, t=kterms: keff_apply(t, H.coupleJ, x), sigma, p, "K")
            q = p + step
            if A_is_sys:
                self.mps[q] = np.tensordot(sigma, self.mps[q], axes=(1, 0))
            else:
                self.mps[q] = np.tensordot(self.mps[q], sigma, axes=(2, 0))
            self.gauges[q] = "Psi"
            self.op_sys_sites.append(op_sys)
        return op_sys

    def propagate(self, dt: float):
        """One time step = forward + backward half sweep (``_mps_cls.py:482-500``)."""
        n = len(self.mps)
        self.sweep(dt, 0, n - 1)
        self.sweep(dt, n - 1, 0)

    # -- observables ----------------------------------------------------------------
    def expectation(self, H: MPOHamiltonian | None = None) -> complex:
        H = self.H if H is None else H
        n = len(self.mps)
        env = self.build_envs(n - 1, 0, H).pop() if n > 1 else zero_site_block()
        terms = terms_for_heff(0, zero_site_block(), env, H, True)
        psi = self.mps[0]
        return complex(np.inner(np.conj(psi).ravel(), heff_apply(terms, H.coupleJ, psi).ravel()))

    def energy(self) -> float:
        return self.expectation().real

    def autocorr(self) -> complex:
        """<Psi(t/2)*|Psi(t/2)> (t/2 trick; ``wavefunction.py:226-257`` with conj=False)."""
        block = np.ones((1, 1), dtype=complex)
        for t in self.mps:
            block = np.einsum("abc,abk->ck", t, np.einsum("ibk,ai->abk", t, block))
        return complex(block[0, 0])

    def norm(self) -> float:
        return float(np.linalg.norm(self.mps[0]))
