"""Thin typed wrapper over the C ABI: torch tensors in, torch tensors out, every op on the GPU.

One ``Engine`` = one ``tdvp_handle_t`` = one GPU / rank.  Nothing here computes on the host: the
methods marshal device pointers and shapes into ``include/tdvp_b200.h`` calls.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from ._lib import GAUGE_A, GAUGE_B, KIND_DIAG, KIND_FULL, Heff2Term, HeffTerm, KeffTerm, check

CDTYPE = torch.complex128


@dataclass
class DeviceCore:
    """An MPO core resident in HBM (reference: ``OperatorCore``, pytdscf/_mpo_cls.py:166-215)."""

    data: torch.Tensor | None  # (wl,d,wr) diagonal or (wl,d,d,wr) full; None = identity gap core
    perm: torch.Tensor | None = None  # full cores: Wp[c,j,i,t] = W[c,i,j,t], made once at upload
    l_id: int = -1  # channel of the incoming MPO bond whose left block is the identity (canonical MPS), -1 = none
    r_id: int = -1  # channel of the outgoing MPO bond whose right block is the identity, -1 = none

    @property
    def kind(self) -> int:
        if self.data is None:
            return _lib.KIND_IDENTITY
        return KIND_DIAG if self.data.dim() == 3 else KIND_FULL

    @property
    def wl(self) -> int:
        return 1 if self.data is None else int(self.data.shape[0])

    @property
    def wr(self) -> int:
        return 1 if self.data is None else int(self.data.shape[-1])


def _ptr(t: torch.Tensor | None):
    return None if t is None else C.c_void_p(t.data_ptr())


def adjoint(M: torch.Tensor) -> torch.Tensor:
    """Conjugate transpose of a 2-D tensor as a contiguous tensor whose MEMORY holds the conjugated values.  ``M.conj()`` only
    sets torch's lazy conjugate bit; ``.T.contiguous()`` materialises it when the transpose forces a copy, but a 1 x n or n x 1
    matrix is already contiguous after ``.T`` and would keep the bit -- the C ABI reads raw memory, so the bit is resolved
    explicitly."""
    return M.conj().T.resolve_conj().contiguous()


def _chk_tensor(t: torch.Tensor, name: str):
    if not (t.is_cuda and t.dtype == CDTYPE and t.is_contiguous()):
        raise TypeError(f"{name} must be a contiguous complex128 CUDA tensor (got {t.dtype}, cuda={t.is_cuda})")


class Engine:
    """Owns a ``tdvp_handle_t`` bound to torch's current stream on ``device``."""

    def __init__(self, device: int | None = None):
        if not torch.cuda.is_available():
            raise RuntimeError("backend='cuda' needs a CUDA device; there is no CPU fallback")
        self.lib = _lib.load_library()
        self.device = torch.cuda.current_device() if device is None else int(device)
        torch.cuda.set_device(self.device)
        self.torch_device = torch.device("cuda", self.device)
        self.stream = torch.cuda.current_stream(self.device)
        h = C.c_void_p()
        rc = self.lib.tdvp_create(self.device, C.c_void_p(self.stream.cuda_stream), C.byref(h))
        if rc != 0:
            raise _lib.TdvpError(rc, "tdvp_create failed")
        self.h = h
        self._keep: list = []  # tensors referenced by descriptors of the call in flight
        self.reorder_mpo_channels = True  # DeviceMPO puts identity-prefix / -suffix channels first / last (see id_channels)

    def close(self):
        if getattr(self, "h", None):
            self.lib.tdvp_destroy(self.h)
            self.h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    # -- uploads ---------------------------------------------------------------------
    def to_device(self, a) -> torch.Tensor:
        return torch.as_tensor(np.ascontiguousarray(a, dtype=np.complex128)).to(self.torch_device)

    def upload_core(self, data) -> DeviceCore:
        if data is None:
            return DeviceCore(None)
        t = self.to_device(data)
        perm = t.permute(0, 2, 1, 3).contiguous() if t.dim() == 4 else None
        return DeviceCore(t, perm)

    def empty(self, *shape) -> torch.Tensor:
        return torch.empty(shape, dtype=CDTYPE, device=self.torch_device)

    # -- descriptors -----------------------------------------------------------------
    def heff_terms(self, terms):
        """terms: iterable of (L | None, DeviceCore | None, R | None, coef)."""
        arr = (HeffTerm * len(terms))()
        for i, (L, core, R, coef) in enumerate(terms):
            t = arr[i]
            t.L = None if L is None else L.data_ptr()
            t.R = None if R is None else R.data_ptr()
            if core is None or core.data is None:
                t.W = None
                t.Wp = None
                t.w_kind = _lib.KIND_IDENTITY
                t.wl = 1 if L is None else int(L.shape[1])
                t.wr = 1 if R is None else int(R.shape[1])
            else:
                t.W = core.data.data_ptr()
                t.Wp = None if core.perm is None else core.perm.data_ptr()
                t.w_kind = core.kind
                t.wl = core.wl
                t.wr = core.wr
                if L is not None and int(L.shape[1]) != core.wl:
                    raise ValueError("left block / core bond dimension mismatch")
                if R is not None and int(R.shape[1]) != core.wr:
                    raise ValueError("right block / core bond dimension mismatch")
                t.id_channels = ((core.l_id + 1) if L is not None else 0) | (((core.r_id + 1) if R is not None else 0) << 16)
            c = complex(coef)
            t.coef_re, t.coef_im = c.real, c.imag
        return arr

    def keff_terms(self, terms):
        """terms: iterable of (L | None, R | None, coef[, (l_id, r_id)]) -- the optional pair names the MPO channels whose
        left / right block is the identity (see ``tdvp_keff_term.id_channels``)."""
        arr = (KeffTerm * len(terms))()
        for i, term in enumerate(terms):
            L, R, coef = term[:3]
            t = arr[i]
            if len(term) > 3 and term[3] is not None and L is not None and R is not None:
                t.id_channels = (term[3][0] + 1) | ((term[3][1] + 1) << 16)
            t.L = None if L is None else L.data_ptr()
            t.R = None if R is None else R.data_ptr()
            if L is not None and R is not None and L.shape[1] != R.shape[1]:
                raise ValueError("K_eff term: MPO bond dimensions of L and R differ")
            t.w = int(L.shape[1]) if L is not None else (int(R.shape[1]) if R is not None else 1)
            c = complex(coef)
            t.coef_re, t.coef_im = c.real, c.imag
        return arr

    def heff2_terms(self, terms):
        """Two-site terms: iterable of (L | None, DeviceCore | None, DeviceCore | None, R | None, coef) -- a None core is the
        identity on that site (a key that acts on the other site only)."""
        arr = (Heff2Term * len(terms))()
        for i, (L, c1, c2, R, coef) in enumerate(terms):
            t = arr[i]
            c1 = None if c1 is None or c1.data is None else c1
            c2 = None if c2 is None or c2.data is None else c2
            t.L = None if L is None else L.data_ptr()
            t.R = None if R is None else R.data_ptr()
            t.wl = 1 if L is None else int(L.shape[1])
            t.wr = 1 if R is None else int(R.shape[1])
            t.wm = c1.wr if c1 is not None else (c2.wl if c2 is not None else 1)
            if c1 is not None and (c1.wl != t.wl or (c2 is not None and c2.wl != c1.wr)) or c2 is not None and c2.wr != t.wr:
                raise ValueError("two-site term: block / core bond dimensions do not match")
            for c, W, Wp, kind in ((c1, "W1", "W1p", "w1_kind"), (c2, "W2", "W2p", "w2_kind")):
                setattr(t, W, None if c is None else c.data.data_ptr())
                setattr(t, Wp, None if c is None or c.perm is None else c.perm.data_ptr())
                setattr(t, kind, _lib.KIND_IDENTITY if c is None else c.kind)
            l_id = c1.l_id if c1 is not None and L is not None else -1
            r_id = c2.r_id if c2 is not None and R is not None else -1
            t.id_channels = (l_id + 1) | ((r_id + 1) << 16)
            c = complex(coef)
            t.coef_re, t.coef_im = c.real, c.imag
        return arr

    # -- contractions ----------------------------------------------------------------
    def heff2_apply(self, terms, theta: torch.Tensor) -> torch.Tensor:
        """out(Dl,d1,d2,Dr) = H2 theta for the two-site terms of ``heff2_terms``."""
        _chk_tensor(theta, "theta")
        Dl, d1, d2, Dr = theta.shape
        out = torch.empty_like(theta)
        arr = self.heff2_terms(terms)
        check(self.h, self.lib.tdvp_heff2_apply(self.h, arr, len(terms), Dl, d1, d2, Dr, _ptr(theta), _ptr(out)))
        return out

    def heff_apply(self, terms, psi: torch.Tensor) -> torch.Tensor:
        _chk_tensor(psi, "psi")
        Dl, d, Dr = psi.shape
        out = torch.empty_like(psi)
        arr = self.heff_terms(terms)
        check(self.h, self.lib.tdvp_heff_apply(self.h, arr, len(terms), Dl, d, Dr, _ptr(psi), _ptr(out)))
        return out

    def keff_apply(self, terms, sigma: torch.Tensor) -> torch.Tensor:
        _chk_tensor(sigma, "sigma")
        Dl, Dr = sigma.shape
        out = torch.empty_like(sigma)
        arr = self.keff_terms(terms)
        check(self.h, self.lib.tdvp_keff_apply(self.h, arr, len(terms), Dl, Dr, _ptr(sigma), _ptr(out)))
        return out

    def env_update(self, gauge: str, bra: torch.Tensor, ket: torch.Tensor, E: torch.Tensor | None,
                   core: DeviceCore | None, out: torch.Tensor | None = None, accumulate: bool = False) -> torch.Tensor:
        _chk_tensor(bra, "bra")
        _chk_tensor(ket, "ket")
        Dl, d, Dr = ket.shape
        g = GAUGE_A if gauge == "A" else GAUGE_B
        has_core = core is not None and core.data is not None
        if gauge == "A":
            w_in = core.wl if has_core else (1 if E is None else int(E.shape[1]))
            w_out = core.wr if has_core else w_in
            D_out = Dr
        else:
            w_in = core.wr if has_core else (1 if E is None else int(E.shape[1]))
            w_out = core.wl if has_core else w_in
            D_out = Dl
        if E is not None and int(E.shape[1]) != w_in:
            raise ValueError("environment block / core bond dimension mismatch")
        if out is None:
            out = self.empty(D_out, w_out, D_out)
            accumulate = False
        check(self.h, self.lib.tdvp_env_update(
            self.h, g, Dl, d, Dr, _ptr(bra), _ptr(ket), _ptr(E), w_in,
            _ptr(core.data) if has_core else None, core.kind if has_core else 0, w_out, _ptr(out), int(accumulate)))
        return out

    # -- Krylov ------------------------------------------------------------------------
    def krylov_expm(self, kind: str, scale: complex, thresh: float, n_warmup: int, conserve_norm: bool,
                    psi: torch.Tensor, *, hterms=None, kterms=None, size_override: int | None = None) -> int:
        """psi <- exp(scale*Op) psi in place; returns the number of Krylov vectors used.  ``size_override``: number of
        elements of the tensor before it was zero-extended (adaptive bond growth, see ``tdvp_set_krylov_size``)."""
        _chk_tensor(psi, "psi")
        if size_override is not None:
            check(self.h, self.lib.tdvp_set_krylov_size(self.h, int(size_override)))
        k = _lib.KRYLOV_ARNOLDI if kind == "arnoldi" else _lib.KRYLOV_LANCZOS_REF
        niter = C.c_int(0)
        scale = complex(scale)
        if hterms is not None:
            Dl, d, Dr = psi.shape
            arr = self.heff_terms(hterms)
            rc = self.lib.tdvp_krylov_expm(self.h, k, scale.real, scale.imag, float(thresh), int(n_warmup),
                                           int(bool(conserve_norm)), arr, None, len(hterms), Dl, d, Dr, _ptr(psi),
                                           C.byref(niter))
        else:
            Dl, Dr = psi.shape
            arr = self.keff_terms(kterms)
            rc = self.lib.tdvp_krylov_expm(self.h, k, scale.real, scale.imag, float(thresh), int(n_warmup),
                                           int(bool(conserve_norm)), None, arr, len(kterms), Dl, 1, Dr, _ptr(psi),
                                           C.byref(niter))
        check(self.h, rc)
        return int(niter.value)

    def krylov_expm2(self, kind: str, scale: complex, thresh: float, n_warmup: int, conserve_norm: bool,
                     theta: torch.Tensor, terms) -> int:
        """theta(Dl,d1,d2,Dr) <- exp(scale*H2) theta in place; returns the number of Krylov vectors used."""
        _chk_tensor(theta, "theta")
        k = _lib.KRYLOV_ARNOLDI if kind == "arnoldi" else _lib.KRYLOV_LANCZOS_REF
        niter = C.c_int(0)
        scale = complex(scale)
        Dl, d1, d2, Dr = theta.shape
        arr = self.heff2_terms(terms)
        check(self.h, self.lib.tdvp_krylov_expm2(self.h, k, scale.real, scale.imag, float(thresh), int(n_warmup),
                                                 int(bool(conserve_norm)), arr, len(terms), Dl, d1, d2, Dr, _ptr(theta),
                                                 C.byref(niter)))
        return int(niter.value)

    def lanczos_eigvec(self, psi: torch.Tensor, hterms, root: int = 0, thresh: float = 1e-9) -> int:
        """psi <- normalised extremal eigenvector of H_eff (improved relaxation); returns the Lanczos dimension."""
        _chk_tensor(psi, "psi")
        Dl, d, Dr = psi.shape
        niter = C.c_int(0)
        arr = self.heff_terms(hterms)
        check(self.h, self.lib.tdvp_lanczos_eigvec(self.h, arr, len(hterms), Dl, d, Dr, _ptr(psi), int(root),
                                                   float(thresh), C.byref(niter)))
        return int(niter.value)

    # -- gauge -------------------------------------------------------------------------
    def regularize_site(self, psi: torch.Tensor) -> torch.Tensor:
        """Floor the small singular values of the (Dl*Dr) x d matricisation (reference ``_site_cls.py:207-252``)."""
        Dl, d, Dr = psi.shape
        M = psi.permute(0, 2, 1).reshape(Dl * Dr, d).contiguous()
        U, s, Vh = self.svd(M)
        eps = 1.0e-4  # SQRT_EPSRHO
        s_reg = np.where(s > eps, s, s + eps * np.exp(-s / eps))
        Us = (U * torch.as_tensor(s_reg, dtype=torch.float64, device=U.device)[None, :]).contiguous()
        return self.zgemm(Us, Vh).reshape(Dl, Dr, d).permute(0, 2, 1).contiguous()

    def qr_shift(self, gauge: str, psi: torch.Tensor, regularize: bool = False):
        """'A': psi -> (A(Dl,d,k), sigma(k,Dr));  'B': psi -> (B(k,d,Dr), sigma(Dl,k))."""
        _chk_tensor(psi, "psi")
        if regularize:
            psi = self.regularize_site(psi)
        Dl, d, Dr = psi.shape
        if gauge == "A":
            if Dl * d < Dr:
                raise ValueError("QR shift needs Dl*d >= Dr")
            site, sigma = self.empty(Dl, d, Dr), self.empty(Dr, Dr)
            g = GAUGE_A
        else:
            if Dr * d < Dl:
                raise ValueError("LQ shift needs Dr*d >= Dl")
            site, sigma = self.empty(Dl, d, Dr), self.empty(Dl, Dl)
            g = GAUGE_B
        check(self.h, self.lib.tdvp_qr_shift(self.h, g, Dl, d, Dr, _ptr(psi), _ptr(site), _ptr(sigma)))
        return site, sigma

    def absorb(self, gauge: str, sigma: torch.Tensor, site: torch.Tensor) -> torch.Tensor:
        """'A': sigma(k,Dl).site(Dl,d,Dr) -> (k,d,Dr);  'B': site(Dl,d,Dr).sigma(Dr,k) -> (Dl,d,k)."""
        _chk_tensor(sigma, "sigma")
        _chk_tensor(site, "site")
        Dl, d, Dr = site.shape
        if gauge == "A":
            k = int(sigma.shape[0])
            out = self.empty(k, d, Dr)
            g = GAUGE_A
        else:
            k = int(sigma.shape[1])
            out = self.empty(Dl, d, k)
            g = GAUGE_B
        check(self.h, self.lib.tdvp_absorb(self.h, g, Dl, d, Dr, k, _ptr(sigma), _ptr(site), _ptr(out)))
        return out

    # -- bond SVD ------------------------------------------------------------------------
    def svd_truncate(self, sigma: torch.Tensor, p: float, keepdim: bool = False, regularize: bool = False):
        """(U, S, Vh, rank) of ``truncate_sigvec(None, sigma, None, p, regularize, keepdim)``."""
        _chk_tensor(sigma, "sigma")
        n = int(sigma.shape[0])
        U, Vh, S = self.empty(n, n), self.empty(n, n), self.empty(n, n)
        rank = C.c_int(0)
        check(self.h, self.lib.tdvp_svd_truncate(self.h, n, int(sigma.shape[1]), _ptr(sigma), float(p), int(keepdim),
                                                 int(regularize), _ptr(U), _ptr(S), _ptr(Vh), C.byref(rank)))
        r = int(rank.value)
        if keepdim:
            return U, S, Vh, r
        return U[:, :r].contiguous(), S.reshape(-1)[: r * r].reshape(r, r), Vh[:r, :].contiguous(), r

    def split2(self, direction: str, theta: torch.Tensor, p: float, Dcap: int, conserve_norm: bool):
        """Truncated split of theta(Dl,d1,d2,Dr): direction "right" -> (A(Dl,d1,r), centre(r,d2,Dr)), "left" ->
        (centre(Dl,d1,r), B(r,d2,Dr)); returns (left, right, s (host float64, all singular values), r)."""
        _chk_tensor(theta, "theta")
        Dl, d1, d2, Dr = theta.shape
        k = max(1, min(int(Dcap), Dl * d1, d2 * Dr))
        left, right = self.empty(Dl * d1 * k), self.empty(k * d2 * Dr)
        s = (C.c_double * min(Dl * d1, d2 * Dr))()
        rank = C.c_int(0)
        g = GAUGE_A if direction == "right" else GAUGE_B
        check(self.h, self.lib.tdvp_split2(self.h, g, Dl, d1, d2, Dr, _ptr(theta), float(p), k, int(bool(conserve_norm)),
                                           _ptr(left), _ptr(right), s, C.byref(rank)))
        r = int(rank.value)
        return (left[: Dl * d1 * r].view(Dl, d1, r), right[: r * d2 * Dr].view(r, d2, Dr), np.array(s[:], dtype=np.float64), r)

    def svd(self, M: torch.Tensor):
        """Thin SVD of a 2-D tensor: (U, s (host float64 array), Vh); wide matrices go through the conjugate transpose."""
        _chk_tensor(M, "M")
        m, n = M.shape
        if m < n:
            U2, s, Vh2 = self.svd(adjoint(M))
            return adjoint(Vh2), s, adjoint(U2)
        U, Vh = self.empty(m, n), self.empty(n, n)
        s = (C.c_double * n)()
        check(self.h, self.lib.tdvp_svd(self.h, m, n, _ptr(M), _ptr(U), s, _ptr(Vh)))
        return U, np.array(s[:], dtype=np.float64), Vh

    def pinv(self, X: torch.Tensor, rcond: float = 1e-13) -> torch.Tensor:
        _chk_tensor(X, "X")
        m, n = X.shape
        out = self.empty(n, m)
        check(self.h, self.lib.tdvp_pinv(self.h, m, n, _ptr(X), float(rcond), _ptr(out)))
        return out

    # -- observables -------------------------------------------------------------------
    def inner(self, bra: torch.Tensor, ket: torch.Tensor, conj: bool = True) -> complex:
        _chk_tensor(bra, "bra")
        _chk_tensor(ket, "ket")
        out = _lib.c128()
        check(self.h, self.lib.tdvp_inner(self.h, bra.numel(), _ptr(bra), _ptr(ket), int(conj), C.byref(out)))
        return complex(out.re, out.im)

    def overlap_site(self, bra: torch.Tensor, ket: torch.Tensor, block: torch.Tensor, conj_bra: bool) -> torch.Tensor:
        Dlb, d, Drb = bra.shape
        Dlk, _, Drk = ket.shape
        out = self.empty(Drb, Drk)
        check(self.h, self.lib.tdvp_overlap_site(self.h, Dlb, Dlk, d, Drb, Drk, _ptr(bra), _ptr(ket), _ptr(block),
                                                 int(conj_bra), _ptr(out)))
        return out

    def zgemm(self, A: torch.Tensor, B: torch.Tensor, transA: int = 0, transB: int = 0, alpha=1.0, beta=0.0,
              C_out: torch.Tensor | None = None) -> torch.Tensor:
        M = A.shape[1] if transA else A.shape[0]
        K = A.shape[0] if transA else A.shape[1]
        N = B.shape[0] if transB else B.shape[1]
        if C_out is None:
            C_out = self.empty(M, N)
        a, b = complex(alpha), complex(beta)
        check(self.h, self.lib.tdvp_zgemm(self.h, transA, transB, M, N, K, a.real, a.imag, _ptr(A), A.shape[1], _ptr(B),
                                          B.shape[1], b.real, b.imag, _ptr(C_out), C_out.shape[1]))
        return C_out

    GEMM_CFGS = {"auto": 0, "big": 1, "small": 2, "tiny": 3, "tma": 4, "tma_tiles": 5}

    def set_gemm_config(self, tile: str = "auto", splitk: int = 0, c_stream: int = 0):
        """Force the GEMM tile configuration / split-K factor / evict-first stores (tests and tuning; see the header)."""
        check(self.h, self.lib.tdvp_set_gemm_config(self.h, self.GEMM_CFGS[tile], int(splitk), int(c_stream)))

    # -- statistics ----------------------------------------------------------------------
    def stats(self) -> dict:
        s, m, f = C.c_ulonglong(0), C.c_ulonglong(0), C.c_double(0.0)
        self.lib.tdvp_get_stats(self.h, C.byref(s), C.byref(m), C.byref(f))
        return {"solves": s.value, "matvecs": m.value, "flops": f.value, "launches": int(self.lib.tdvp_launch_count())}

    def reset_stats(self):
        self.lib.tdvp_reset_stats(self.h)

    def gemm_profile(self, enable: bool, reset: bool = False) -> dict:
        """Collect the per-launch GEMM timings recorded so far, then switch recording on/off."""
        ms, fl, n = C.c_double(0.0), C.c_double(0.0), C.c_ulonglong(0)
        self.lib.tdvp_gemm_profile(int(enable), int(reset), C.byref(ms), C.byref(fl), C.byref(n))
        return {"ms": ms.value, "flops": fl.value, "launches": n.value}

    def profile_breakdown(self) -> dict:
        """Per-label totals (ms, flops, launches) of everything recorded since the last reset."""
        import json

        buf = C.create_string_buffer(1 << 16)
        self.lib.tdvp_profile_json(buf, len(buf))
        return json.loads(buf.value.decode())
