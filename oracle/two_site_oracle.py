"""CPU oracle of two-site TDVP -- TEST INFRASTRUCTURE, NOT A PRODUCT PATH.

The reference (PyTDSCF 1.3.3) has no two-site TDVP, so there is no golden run to pin this against.  It is restated from
pieces of ``oracle/tdvp_oracle.py`` that ARE pinned to the reference: the einsum H_eff contraction (one more core),
``sil_reference`` / ``sia_reference``, the environment bookkeeping (``renormalize``, ``terms_for_heff``), and the
cumulative singular-value truncation rule of ``truncate_bond`` (``truncate_sigvec``).  At full bond dimension the composed
algorithm has an exact answer, dense ``expm``, which tests/test_two_site_cpu.py checks.  Only ``tests/`` imports it.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np

from oracle import tdvp_oracle as orc


def heff2_term(L, core1, core2, R, theta: np.ndarray) -> np.ndarray:
    """One MPO term of the two-site H_eff: out[a,i,k,r] = sum L[a,c,b] W1[c,i,j,t] W2[t,k,l,u] R[r,u,s] theta[b,j,l,s].

    ``core1`` / ``core2``: SiteCore or ``None`` (identity on that site; its MPO bonds have dimension 1, so the blocks'
    channel sums next to it run over a single channel).  The reference has no two-site path; this is the one-site
    ``heff_term`` with one more core."""
    W1 = None if core1 is None else core1.data
    W2 = None if core2 is None else core2.data
    ops, lhs = [theta], ["bjls"]
    a, i, k, r = "b", "j", "l", "s"
    if L is not None:
        ops.append(L)
        lhs.append("acb")
        a = "a"
    if W1 is not None:
        ops.append(W1)
        if W1.ndim == 3:
            lhs.append("cjt")
        else:
            lhs.append("cijt")
            i = "i"
    if W2 is not None:
        ops.append(W2)
        if W2.ndim == 3:
            lhs.append("tlu")
        else:
            lhs.append("tklu")
            k = "k"
    if R is not None:
        ops.append(R)
        lhs.append("rus")
        r = "r"
    if len(ops) == 1:
        return theta
    return orc._einsum(",".join(lhs) + "->" + a + i + k + r, *ops)


def heff2_apply(terms: list, theta: np.ndarray) -> np.ndarray:
    """Sum of ``coef * heff2_term`` over ``terms`` = [(L, core1, core2, R, coef)] in list order."""
    out = None
    for L, c1, c2, R, coef in terms:
        add = heff2_term(L, c1, c2, R, theta)
        if complex(coef) != 1.0:
            add = add * complex(coef)
        out = add.copy() if out is None else out + add
    return out


def split_two_site(theta: np.ndarray, direction: str, p: float, Dcap: int, conserve_norm: bool):
    """Truncated SVD split of theta(Dl, d1, d2, Dr) -> (left(Dl,d1,r), right(r,d2,Dr), s, r).

    Rank r = min(r_p, Dcap) >= 1, r_p the smallest index whose cumulative singular-VALUE sum reaches (1 - p) of the
    total (``truncate_bond``'s rule); ``conserve_norm`` rescales the kept values to the norm of all of them.
    "right": left = U (gauge A), right = diag(s) Vh (centre); "left": left = U diag(s) (centre), right = Vh (gauge B)."""
    Dl, d1, d2, Dr = theta.shape
    U, s, Vh = np.linalg.svd(theta.reshape(Dl * d1, d2 * Dr), full_matrices=False)
    cs = np.cumsum(s)
    rp = len(s)
    if cs[-1] > 0.0:
        hit = np.nonzero(cs / cs[-1] >= 1.0 - p)[0]
        rp = int(hit[0]) + 1 if len(hit) else len(s)
    r = max(1, min(rp, int(Dcap), len(s)))
    sk = s[:r].copy()
    if conserve_norm:
        kept = float(np.sqrt(np.sum(sk**2)))
        if kept > 0.0:
            sk = sk * (float(np.sqrt(np.sum(s**2))) / kept)
    if direction == "right":
        left, right = U[:, :r], sk[:, None] * Vh[:r]
    elif direction == "left":
        left, right = U[:, :r] * sk[None, :], Vh[:r]
    else:
        raise ValueError(direction)
    return (np.ascontiguousarray(left).reshape(Dl, d1, r), np.ascontiguousarray(right).reshape(r, d2, Dr), s, r)


def terms_for_heff2(p: int, Lb: dict, Rb: dict, H: orc.MPOHamiltonian) -> list:
    """Terms of the two-site H_eff of sites (p, p+1): [(L, core1, core2, R, coef)] -- coupleJ on the overlap blocks, the
    summed blocks, then every key acting on p or p+1 (keys of p first, in calc_point order)."""
    Lo, Ro = orc._ovlp_operand(Lb), orc._ovlp_operand(Rb)
    terms = []
    if H.coupleJ != 0.0:
        terms.append((Lo, None, None, Ro, H.coupleJ))
    if "summed" in Lb:
        terms.append((Lb["summed"], None, None, Ro, 1.0))
    if "summed" in Rb:
        terms.append((Lo, None, None, Rb["summed"], 1.0))
    c1 = {c.key: c for c in H.calc_point[p]}
    c2 = {c.key: c for c in H.calc_point[p + 1]}
    for key in list(c1) + [k for k in c2 if k not in c1]:
        terms.append((Lb.get(key, Lo), c1.get(key), c2.get(key), Rb.get(key, Ro), 1.0))
    return terms


@dataclass
class TwoSiteOracle(orc.TDVPOracle):
    """``TDVPOracle`` with the two-site sweep.  Trace entries: ("H2", pair, niter) for the pair solves and ("H1b", site,
    niter) for the backward-in-time one-site solves; warm-up keys ("pair", p) / ("site", q)."""

    bond_dim: int | None = None  # bond-dimension cap (None: only the rank of the matricisation)
    p_svd: float = 1.0e-07  # truncation weight of the split

    def _dcap(self, p: int) -> int:
        dims = [t.shape[1] for t in self.mps]
        cap = min(math.prod(dims[: p + 1]), math.prod(dims[p + 1 :]))
        return cap if self.bond_dim is None else min(cap, int(self.bond_dim))

    def _expm_key(self, key, kind: str, index: int, sign: complex, dt: float, matvec, x):
        solver = orc.sia_reference if self.integrator == "arnoldi" else orc.sil_reference
        y, n = solver(sign * (dt / 2), matvec, x, self.thresh, last_niter=self.niter.get(key, 0),
                      conserve_norm=self.conserve_norm)
        self.niter[key] = n
        self.trace.append((kind, index, n))
        return y

    def sweep_two_site(self, dt: float, forward: bool, envs: list | None = None) -> list:
        """One two-site half sweep.  Forward (centre at 0, the rest B), pairs p = 0 .. n-2: theta = psi_p B_{p+1},
        theta <- exp(-i H2 dt/2) theta, split "right" into A_p and psi_{p+1}, then (p < n-2) psi_{p+1} <- exp(+i H1 dt/2)
        psi_{p+1}.  Backward mirrors it for p = n-2 .. 0 with split "left" and the one-site step on psi_p for p > 0.
        ``envs``: the far-side blocks (as the previous half sweep returns them); returns the near-side blocks it built."""
        n = len(self.mps)
        H = self.H
        if envs is None:
            envs = self.build_envs(n - 1, 1) if forward else self.build_envs(0, n - 2)
        done = [orc.zero_site_block()]
        for p in range(n - 1) if forward else range(n - 2, -1, -1):
            if forward:
                Lb, Rb = done[-1], envs.pop()
            else:
                Lb, Rb = envs.pop(), done[-1]
            theta = np.tensordot(self.mps[p], self.mps[p + 1], axes=(2, 0))
            terms = terms_for_heff2(p, Lb, Rb, H)
            theta = self._expm_key(("pair", p), "H2", p, -1.0j, dt, lambda x, t=terms: heff2_apply(t, x), theta)
            left, right, _s, _r = split_two_site(theta, "right" if forward else "left", self.p_svd, self._dcap(p),
                                                 self.conserve_norm)
            self.mps[p], self.mps[p + 1] = left, right
            if forward:
                self.gauges[p], self.gauges[p + 1] = "A", "Psi"
                if p < n - 2:
                    Lb = orc.renormalize(p, left, "A", Lb, H, True)
                    done.append(Lb)
                    t1 = orc.terms_for_heff(p + 1, Lb, Rb, H, True)
                    self.mps[p + 1] = self._expm_key(("site", p + 1), "H1b", p + 1, +1.0j, dt,
                                                     lambda x, t=t1: orc.heff_apply(t, H.coupleJ, x), right)
            else:
                self.gauges[p], self.gauges[p + 1] = "Psi", "B"
                if p > 0:
                    Rb = orc.renormalize(p + 1, right, "B", Rb, H, False)
                    done.append(Rb)
                    t1 = orc.terms_for_heff(p, Rb, Lb, H, False)
                    self.mps[p] = self._expm_key(("site", p), "H1b", p, +1.0j, dt,
                                                 lambda x, t=t1: orc.heff_apply(t, H.coupleJ, x), left)
        return done

    def propagate_two_site(self, dt: float):
        """One two-site time step: forward + backward half sweep, each with dt/2 per local solve."""
        if len(self.mps) < 2:
            raise ValueError("two-site TDVP needs at least two sites")
        self.sweep_two_site(dt, False, self.sweep_two_site(dt, True))

    def bonddim(self) -> list[int]:
        return [t.shape[2] for t in self.mps[:-1]]
