"""Two-site TDVP on the device: the bond dimensions follow the state, from a Hartree product up to the model's ``bond_dim``.

One time step is a forward and a backward half sweep with dt/2 per local solve (the one-site step's structure):
  forward, centre at 0 and the rest B, pairs p = 0 .. n-2:
    theta = psi_p B_{p+1}                          one GEMM
    theta <- exp(-i H2(p, p+1) dt/2) theta         tdvp_krylov_expm2 on the two-site H_eff
    theta -> A_p, psi_{p+1}                        tdvp_split2 "right": truncated SVD
    left block of p                                tdvp_env_update (renormalize_op_psite)
    psi_{p+1} <- exp(+i H1(p+1) dt/2) psi_{p+1}    p < n-2 only, one-site H_eff
  backward mirrors it for p = n-2 .. 0 with split "left" and the one-site step on psi_p for p > 0.  The last pair gets two
  consecutive half steps (not merged), as the last site of the one-site sweep does.

The blocks the backward sweep needs are the ones the forward sweep built; each time step rebuilds the right blocks once
at its start.  Krylov warm-up history: keys ("pair", p) and ("site", q), apart from the one-site keys; the trace records
(TRACE_PAIR, p, niter) and (TRACE_SITE_BACK, q, niter).  The arithmetic is Engine calls; Python does bookkeeping only.
"""
from __future__ import annotations

import dataclasses
import math

from ._mps_cuda import DeviceMPO, MPSCoefCuda, SiteCoef

TRACE_PAIR, TRACE_SITE_BACK = 2, 3


def bond_cap(mps: MPSCoefCuda, p: int, bond_dim: int) -> int:
    """Largest bond between sites p and p+1: min(bond_dim, prod of the dims left of it, prod of the dims right of it) --
    the static rule of ``bond_dims``; bond_dim <= 0 means no cap beyond the matricisation ranks."""
    dims = [s.shape[1] for s in mps.sites]
    cap = min(math.prod(dims[: p + 1]), math.prod(dims[p + 1:]))
    return cap if bond_dim <= 0 else min(cap, bond_dim)


def operators_for_pair(mps: MPSCoefCuda, p: int, Lb: dict, Rb: dict, H: DeviceMPO) -> list:
    """Two-site H_eff terms of sites (p, p+1): [(L, core_p | None, core_{p+1} | None, R, coef)] in the order of the
    oracle's ``terms_for_heff2``: coupleJ (identity operator), the summed blocks, then every key acting on p or p+1."""
    Lo, Ro = mps._ovlp(Lb), mps._ovlp(Rb)
    terms = []
    if H.coupleJ != 0.0:
        terms.append((Lo, None, None, Ro, H.coupleJ))
    if "summed" in Lb:
        terms.append((Lb["summed"], None, None, Ro, 1.0))
    if "summed" in Rb:
        terms.append((Lo, None, None, Rb["summed"], 1.0))
    off = mps.site_offset
    c1 = {t.key: t.core for t in H.calc_point[p + off]}
    c2 = {t.key: t.core for t in H.calc_point[p + 1 + off]}
    for key in list(c1) + [k for k in c2 if k not in c1]:
        k1, k2 = c1.get(key), c2.get(key)
        # the identity-channel promise holds only while the overlap blocks are identities (canonical sites)
        if k1 is not None and k1.l_id >= 0 and Lo is not None:
            k1 = dataclasses.replace(k1, l_id=-1)
        if k2 is not None and k2.r_id >= 0 and Ro is not None:
            k2 = dataclasses.replace(k2, r_id=-1)
        terms.append((Lb.get(key, Lo), k1, k2, Rb.get(key, Ro), 1.0))
    return terms


def _solve(mps: MPSCoefCuda, cfg, dt: float, sign: complex, x, key, kind: int, index: int, *, pair_terms=None, hterms=None):
    eng = mps.eng
    n_warm = mps._n_warmup(x.numel(), key)
    y = x.clone()
    if pair_terms is not None:
        niter = eng.krylov_expm2(cfg.integrator, sign * (dt / 2), cfg.thresh_exp, n_warm, cfg.conserve_norm, y, pair_terms)
    else:
        niter = eng.krylov_expm(cfg.integrator, sign * (dt / 2), cfg.thresh_exp, n_warm, cfg.conserve_norm, y, hterms=hterms)
    mps.niter_krylov[key] = niter
    if mps.record_trace:
        mps.trace.append((kind, index, niter))
    return y


def half_sweep(mps: MPSCoefCuda, H: DeviceMPO, dt: float, cfg, forward: bool, envs: list | None = None) -> list:
    """One two-site half sweep (see the module docstring).  ``envs``: far-side blocks; returns the near-side blocks."""
    eng, sb, n = mps.eng, mps.sites, mps.nsite
    if envs is None:
        envs = mps.construct_op_sites(n - 1, 1, H) if forward else mps.construct_op_sites(0, n - 2, H)
    done = [mps.construct_op_zerosite()]
    for p in range(n - 1) if forward else range(n - 2, -1, -1):
        mps.site_now = p
        if forward:
            Lb, Rb = done[-1], envs.pop()
        else:
            Lb, Rb = envs.pop(), done[-1]
        a, d1, D = sb[p].shape
        _, d2, e = sb[p + 1].shape
        theta = eng.zgemm(sb[p].data.reshape(a * d1, D), sb[p + 1].data.reshape(D, d2 * e)).reshape(a, d1, d2, e)
        theta = _solve(mps, cfg, dt, -1.0j, theta, ("pair", p), TRACE_PAIR, p, pair_terms=operators_for_pair(mps, p, Lb, Rb, H))
        left, right, _s, _r = eng.split2("right" if forward else "left", theta, cfg.two_site_p_svd,
                                         bond_cap(mps, p, cfg.bond_dim), cfg.conserve_norm)
        if forward:
            sb[p], sb[p + 1] = SiteCoef(left, "A", p), SiteCoef(right, "Psi", p + 1)
            if p < n - 2:
                Lb = mps.renormalize_op_psite(p, Lb, H, True)
                done.append(Lb)
                hterms = mps.operators_for_superH(p + 1, Lb, Rb, H, True)
                sb[p + 1] = SiteCoef(_solve(mps, cfg, dt, +1.0j, right, ("site", p + 1), TRACE_SITE_BACK, p + 1, hterms=hterms),
                                     "Psi", p + 1)
        else:
            sb[p], sb[p + 1] = SiteCoef(left, "Psi", p), SiteCoef(right, "B", p + 1)
            if p > 0:
                Rb = mps.renormalize_op_psite(p + 1, Rb, H, False)
                done.append(Rb)
                hterms = mps.operators_for_superH(p, Rb, Lb, H, False)
                sb[p] = SiteCoef(_solve(mps, cfg, dt, +1.0j, left, ("site", p), TRACE_SITE_BACK, p, hterms=hterms), "Psi", p)
    return done


def propagate_two_site(mps: MPSCoefCuda, stepsize: float, H: DeviceMPO, cfg):
    """One two-site time step; the centre is back at site 0 afterwards."""
    if mps.nsite < 2:
        raise ValueError("two-site TDVP needs a chain of at least two sites")
    half_sweep(mps, H, stepsize, cfg, False, half_sweep(mps, H, stepsize, cfg, True))
    mps.op_sys_sites = None   # the one-site sweep's cached blocks belong to the old bonds
