"""MPS coefficient object of ``backend="cuda"``: one-site projector-splitting TDVP with every tensor in HBM.

Mirrors the reference's serial MPO path (file:line relative to the PyTDSCF tree):
  alloc_random / initial MPS       pytdscf/_mps_mpo.py:55-133 ; pytdscf/_mps_cls.py:2616-2703
  construct_op_zerosite            pytdscf/_mps_mpo.py:364-419
  renormalize_op_psite             pytdscf/_mps_mpo.py:421-696
  operators_for_superH / superK    pytdscf/_mps_mpo.py:698-858, 860-1021
  propagate / propagate_along_sweep   pytdscf/_mps_cls.py:452-503, 798-1014
  exp_superH/K_propagation_direct  pytdscf/_mps_cls.py:1016-1170
  trans_next_psite_AsigmaB/APsiB   pytdscf/_mps_cls.py:1798-1850, 1172-1206
  expectation / autocorr / norm    pytdscf/_mps_cls.py:540-612, 706-716 ; pytdscf/wavefunction.py:226-257

The Python here is bookkeeping only (which block meets which core, per-site Krylov history, environment
hand-over between sweeps); all arithmetic is ``Engine`` calls into libtdvp_b200 (no NumPy on tensors).
"""
from __future__ import annotations

import math
import dataclasses
from dataclasses import dataclass

import numpy as np
import torch

from ._engine import DeviceCore, Engine
from .hamiltonian_cls import TensorHamiltonian

KRYLOV_CAP = 20


@dataclass
class SiteCoef:
    """Site tensor + gauge label (reference: ``pytdscf/_site_cls.py:27-136``); ``data`` lives on the GPU."""

    data: torch.Tensor
    gauge: str
    isite: int

    @property
    def shape(self):
        return tuple(self.data.shape)

    def numpy(self) -> np.ndarray:
        return self.data.cpu().numpy()

    def __array__(self, dtype=None, copy=None):
        return self.numpy()


@dataclass
class Block:
    """Environment block (bra, mpo, ket) = (D, w, D); identity blocks carry only their size."""

    data: torch.Tensor | None
    is_identity: bool = False
    dim: int = 1


@dataclass
class DeviceTerm:
    key: tuple
    core: DeviceCore
    is_left: bool
    is_right: bool


def identity_channels(cores: list[np.ndarray]) -> tuple[list[int], list[int]]:
    """For the cores of one MPO term return ``(pre, suf)``: ``pre[k]`` = channel of the bond LEFT of core k that carries
    nothing but identity operators from the left end (its left environment block is <A|A> = 1 for canonical tensors),
    ``suf[k]`` = channel of the bond RIGHT of core k that carries only identities up to the right end; -1 = none.
    Exact comparisons only: a channel qualifies when its single incoming (outgoing) block is exactly the unit matrix."""
    n = len(cores)

    def is_unit(b: np.ndarray) -> bool:
        return bool(np.array_equal(b, np.ones_like(b))) if b.ndim == 1 else bool(np.array_equal(b, np.eye(b.shape[0])))

    bond = [-1] * (n + 1)           # bond[k]: identity-prefix channel of the bond left of core k
    bond[0] = 0 if cores[0].shape[0] == 1 else -1
    for k, W in enumerate(cores):
        if bond[k] < 0:
            break
        for t in range(W.shape[-1]):
            col = W[..., t]
            nz = [c for c in range(W.shape[0]) if np.any(col[c] != 0)]
            if nz == [bond[k]] and is_unit(col[bond[k]]):
                bond[k + 1] = t
                break
    dnob = [-1] * (n + 1)           # dnob[k]: identity-suffix channel of the bond left of core k (right of core k-1)
    dnob[n] = 0 if cores[-1].shape[-1] == 1 else -1
    for k in range(n - 1, -1, -1):
        W = cores[k]
        if dnob[k + 1] < 0:
            break
        for c in range(W.shape[0]):
            row = W[c]
            nz = [t for t in range(W.shape[-1]) if np.any(row[..., t] != 0)]
            if nz == [dnob[k + 1]] and is_unit(row[..., dnob[k + 1]]):
                dnob[k] = c
                break
    return bond[:n], dnob[1:]


def direct_sum_mpo(core_lists: list[list[np.ndarray]]) -> list[np.ndarray]:
    """Direct sum of full-length MPOs: ONE MPO whose bond space is the disjoint union of the inputs' bond spaces
    (block-diagonal cores, a row of blocks on the first site and a column on the last), i.e. the operator sum.  Diagonal
    (3-index) cores are expanded to 4-index ones."""
    n = len(core_lists[0])
    full = []
    for cores in core_lists:
        row = []
        for W in cores:
            W = np.asarray(W, dtype=np.complex128)
            if W.ndim == 3:
                d = W.shape[1]
                F = np.zeros((W.shape[0], d, d, W.shape[2]), dtype=np.complex128)
                idx = np.arange(d)
                F[:, idx, idx, :] = W
                W = F
            row.append(W)
        full.append(row)
    out = []
    for k in range(n):
        blocks = [row[k] for row in full]
        d = blocks[0].shape[1]
        wl = 1 if k == 0 else sum(b.shape[0] for b in blocks)
        wr = 1 if k == n - 1 else sum(b.shape[3] for b in blocks)
        W = np.zeros((wl, d, d, wr), dtype=np.complex128)
        a = c = 0
        for b in blocks:
            la, lc = (0 if k == 0 else a), (0 if k == n - 1 else c)
            W[la:la + b.shape[0], :, :, lc:lc + b.shape[3]] += b
            a += b.shape[0]
            c += b.shape[3]
        out.append(W)
    return out


class DeviceMPO:
    """MPO cores of a ``TensorHamiltonian`` uploaded to HBM once (complex128; float cores are widened).

    ``merge_terms``: combine all MPO keys that span the whole chain into one direct-sum MPO.  The operator is the same sum;
    H_eff / K_eff / the environment updates then issue one GEMM chain instead of one per key.  Worth it only where a sweep
    is bound by kernel LAUNCHES (D <= 64: BASELINE configs 1 and 2 carry a potential and a kinetic MPO): the block-diagonal
    cores make stage 2 do (w_1 + w_2)^2 d^2 work instead of w_1^2 d + w_2^2 d^2, which would cost 10-15 % of a step at
    D >= 256, and the order of the term sum (hence rounding) differs from the reference's."""

    def __init__(self, eng: Engine, ham: TensorHamiltonian, merge_terms: bool = False):
        mpo = ham.mpo[0][0]
        self.coupleJ = complex(ham.coupleJ[0][0])
        self.nsite = mpo.nsite
        self.calc_point: list[list[DeviceTerm]] = [[] for _ in range(mpo.nsite)]
        self.bond_ids: dict = {}   # (key, bond b between sites b-1 and b) -> (prefix channel, suffix channel)
        # per key the cores as the site lists hold them NOW (a Liouville sub-space projection, ``project_subspace``, has
        # already cut their physical indices there), in site order
        by_key: dict = {}
        for cps in mpo.calc_point:
            for c in cps:
                by_key.setdefault(c.key, []).append((c.psite, c.data))
        term_list = []          # (key, sites, cores)
        for key, lst in by_key.items():
            if any(isinstance(d, int) for _, d in lst):
                raise NotImplementedError(
                    f"MPO key {key} skips a site: identity gap cores fail in the reference's H_eff apply "
                    "as well (pytdscf/_contraction.py:1067); give full-length cores instead")
            term_list.append((key, [s for s, _ in lst], [np.asarray(d) for _, d in lst]))
        if merge_terms:
            whole = [t for t in term_list if t[1] == list(range(mpo.nsite))]
            if len(whole) >= 2 and mpo.nsite >= 2:
                merged_key = ("direct_sum",) + tuple(t[0] for t in whole)
                rest = [t for t in term_list if t[1] != list(range(mpo.nsite))]
                term_list = [(merged_key, list(range(mpo.nsite)), direct_sum_mpo([t[2] for t in whole]))] + rest
        self.merged = merge_terms and any(isinstance(t[0], tuple) and t[0][:1] == ("direct_sum",) for t in term_list)
        for key, sites, cores in term_list:
            pre, suf = identity_channels(cores)
            # Re-order the channels of every internal bond so that the identity-prefix channel comes first and the
            # identity-suffix channel last (the same permutation on the right index of core k-1 and the left index of
            # core k leaves the operator unchanged): the shortcut GEMMs then skip a contiguous end of the channel range.
            # Engines that implement the shortcut ask for it (``reorder_mpo_channels``); the order of the channel sum
            # changes rounding, so test engines that compare bit-for-bit with the reference keep the given order.
            for k in range(1, len(cores) if getattr(eng, "reorder_mpo_channels", False) else 0):
                w = cores[k].shape[0]
                a, z = pre[k], suf[k - 1]
                if z == a:
                    z = -1
                order = ([a] if a >= 0 else []) + [c for c in range(w) if c != a and c != z] + ([z] if z >= 0 else [])
                if order != list(range(w)):
                    cores[k - 1] = np.ascontiguousarray(np.take(cores[k - 1], order, axis=-1))
                    cores[k] = np.ascontiguousarray(np.take(cores[k], order, axis=0))
            pre, suf = identity_channels(cores)
            lo, hi = min(sites), max(sites)
            for k, site in enumerate(sites):
                dc = eng.upload_core(cores[k])
                dc.l_id, dc.r_id = pre[k], suf[k]
                self.calc_point[site].append(DeviceTerm(key, dc, site == lo, site == hi))
                if k > 0 and sites[k - 1] == site - 1:
                    self.bond_ids[(key, site)] = (pre[k], suf[k - 1])


def bond_dims(dims: list[int], isite: int, m: int) -> tuple[int, int]:
    """Static bond-dimension rule (``LatticeInfo.get_bond_dim``, _mps_cls.py:2616-2631)."""
    n = len(dims)
    dim_left = 1 if isite == 0 else min(m, math.prod(dims[:isite]))
    dim_right = 1 if isite == n - 1 else min(m, math.prod(dims[isite + 1:]))
    dc = dims[isite]
    return min(dim_left, dc * dim_right, m), min(dim_left * dc, dim_right, m)


# ---------------------------------------------------------------------------------------------------------
# canonicalisation helpers on device tensors (_mps_cls.py:3470-3630)
# ---------------------------------------------------------------------------------------------------------
def canonicalizeA(eng, sb: list):
    sval = None
    for i, coef in enumerate(sb):
        if sval is not None:
            coef.data = eng.absorb("A", sval, coef.data)
        coef.gauge = "Psi"
        if i != len(sb) - 1:
            coef.data, sval = eng.qr_shift("A", coef.data)
            coef.gauge = "A"


def canonicalizeB(eng, sb: list):
    sval = None
    for i, coef in enumerate(sb[::-1]):
        if sval is not None:
            coef.data = eng.absorb("B", sval, coef.data)
        coef.gauge = "Psi"
        if i != len(sb) - 1:
            coef.data, sval = eng.qr_shift("B", coef.data)
            coef.gauge = "B"


def cc2_a_lambda_b(eng, left: SiteCoef, right: SiteCoef) -> np.ndarray:
    """SVD of the two-site tensor: left <- U (gauge A), right <- Vh (gauge B); returns the singular values (host)."""
    a, b, c = left.data.shape
    _, d, e = right.data.shape
    two = eng.zgemm(left.data.reshape(a * b, c).contiguous(), right.data.reshape(c, d * e).contiguous())
    U, lam, Vh = eng.svd(two)
    left.data = U[:, :c].contiguous().reshape(a, b, c)
    left.gauge = "A"
    right.data = Vh[:c, :].contiguous().reshape(c, d, e)
    right.gauge = "B"
    return np.asarray(lam[:c])


def canonicalize(eng, sb: list, center: int, incremental: bool = False):
    n = len(sb)
    if n == 1:
        return
    if incremental:
        cur = [i for i, s in enumerate(sb) if s.gauge == "Psi"]
        if len(cur) != 1:
            raise ValueError("canonicalize(incremental): exactly one Psi site expected")
        cur = cur[0]
        if cur == center:
            return
        if cur < center:
            canonicalizeA(eng, sb[cur:center + 1])
        else:
            canonicalizeB(eng, sb[center:cur + 1])
        return
    canonicalizeB(eng, sb[center:])
    if center == 0:
        return
    canonicalizeA(eng, sb[:center])
    lam = cc2_a_lambda_b(eng, sb[center - 1], sb[center])
    lam_t = torch.as_tensor(lam, dtype=torch.float64, device=sb[center].data.device)
    sb[center].data = (lam_t[:, None, None] * sb[center].data).contiguous()
    sb[center].gauge = "Psi"



def oversize_bonds(sb: list) -> list[int]:
    """Bonds (index of the site on their left) larger than the matricisations next to them allow: D_r > D_l d of the left
    site or D_l > d D_r of the right one.  ``LatticeInfo.get_bond_dim`` (_mps_cls.py:2616-2631) never produces such bonds,
    hand-made site tensors can."""
    bad = []
    for i in range(len(sb) - 1):
        a, d, D = sb[i].data.shape
        _, d2, e = sb[i + 1].data.shape
        if D > a * d or D > d2 * e:
            bad.append(i)
    return bad


def compress_oversize_bonds(eng, sb: list, center: int = 0) -> bool:
    """Exact compression of every bond that exceeds the rank its neighbours can carry, then re-canonicalisation around
    ``center``.  The reference never sees such bonds as an error: its economic QR in ``gauge_trf`` (_site_cls.py:138-292)
    silently shrinks a bond to min(rows, columns) at the first sweep.  Here ``tdvp_qr_shift`` factors tall matrices only, so
    explicit site tensors (``Simulator.set_initial_mps``, own-format checkpoints) are brought to the reference's bond rule once,
    at upload: thin SVDs of the offending matricisations (U to one side, S Vh folded into the neighbour) -- the represented
    state is unchanged to rounding.  Returns True when something was compressed."""
    if not oversize_bonds(sb):
        return False
    for _ in range(len(sb) + 1):                 # bonds only shrink: at most nsite passes
        bad = oversize_bonds(sb)
        if not bad:
            break
        for i in bad:
            L, R = sb[i].data, sb[i + 1].data
            a, d, D = L.shape
            _, d2, e = R.shape
            if D > a * d:                        # left matricisation (a d) x D is wide: rank <= a d
                U, sv, Vh = eng.svd(L.reshape(a * d, D).contiguous())
                k = U.shape[1]
                scale = torch.as_tensor(np.asarray(sv[:k]), dtype=torch.float64, device=U.device)
                sb[i].data = U.contiguous().reshape(a, d, k)
                sb[i + 1].data = eng.zgemm((scale[:, None] * Vh[:k, :]).contiguous(), R.reshape(D, d2 * e).contiguous()).reshape(k, d2, e)
            elif D > d2 * e:                     # right matricisation D x (d2 e) is tall: rank <= d2 e
                U, sv, Vh = eng.svd(R.reshape(D, d2 * e).contiguous())
                k = Vh.shape[0]
                scale = torch.as_tensor(np.asarray(sv[:k]), dtype=torch.float64, device=U.device)
                sb[i + 1].data = Vh.contiguous().reshape(k, d2, e)
                sb[i].data = eng.zgemm(L.reshape(a * d, D).contiguous(), (U[:, :k] * scale[None, :]).contiguous()).reshape(a, d, k)
    if oversize_bonds(sb):
        raise RuntimeError("compress_oversize_bonds did not reach the bond-dimension rule")
    canonicalize(eng, sb, center, incremental=False)
    return True


class MPSCoefCuda:
    """Device-resident MPS in mixed-canonical form with the orthogonality centre at site 0 between steps."""

    def __init__(self, eng: Engine, cores: list[torch.Tensor], gauges: list[str] | None = None):
        self.eng = eng
        n = len(cores)
        gauges = gauges or ["Psi"] + ["B"] * (n - 1)
        self.superblock_states = [[SiteCoef(c, g, i) for i, (c, g) in enumerate(zip(cores, gauges, strict=True))]]
        self.nsite = n
        self.nstate = 1
        self.op_sys_sites: list | None = None
        self.niter_krylov: dict[int, int] = {}   # shared by the H and K solves of a site (SURVEY F3)
        self.trace: list[tuple[int, int, int]] = []  # (0=H|1=K, site, niter)
        self.record_trace = False
        self.site_offset = 0   # global index of local site 0 (site-parallel segments share one global MPO)
        self.site_now = 0      # reference: helper._Debug.site_now, the key of the Krylov warm-up history
        self.subspace: dict[int, tuple[int, tuple[int, ...]]] = {}   # Liouville sub-space sites: site -> (full d, kept indices)

    @classmethod
    def from_user_cores(cls, eng: Engine, cores: list, gauges: list[str] | None = None) -> "MPSCoefCuda":
        """Explicit site tensors (``Simulator.set_initial_mps``, checkpoints): uploaded as given; bonds beyond the reference's
        bond-dimension rule are compressed exactly and the chain is re-canonicalised around its centre (see
        ``compress_oversize_bonds``)."""
        mps = cls(eng, [c if isinstance(c, torch.Tensor) else eng.to_device(np.ascontiguousarray(c, dtype=np.complex128)) for c in cores], gauges)
        sb = mps.sites
        centres = [i for i, s in enumerate(sb) if s.gauge == "Psi"]
        compress_oversize_bonds(eng, sb, centres[0] if len(centres) == 1 else 0)
        return mps

    # ------------------------------------------------------------------------------------------
    @classmethod
    def alloc_random(cls, eng: Engine, model) -> "MPSCoefCuda":
        """Zero-padded Hartree product, right-canonicalised by LQ sweeps on the device (despite the reference's
        name nothing is random).  The LQ uses the same Householder conventions as LAPACK, so the null-space
        completion of the padded tensors matches the reference (tests/test_gpu_kernels.py)."""
        weights, scale, m = model.initial_core_weights()
        dims = [len(model.get_primbas(0, i)) for i in range(model.get_ndof())]
        n = len(dims)
        host = []
        for i in range(n):
            ml, mr = bond_dims(dims, i, m)
            data = np.zeros((1 if i == 0 else ml, dims[i], 1 if i == n - 1 else mr), dtype=np.complex128)
            w = np.array(weights[i], dtype=np.complex128)
            if w.ndim == 1:
                data[0, :, 0] = w
                if model.space == "hilbert":
                    data[0, :, 0] /= np.linalg.norm(w)
                else:
                    q = math.isqrt(dims[i])
                    data[0, :, 0] /= np.trace(w.reshape(q, q))
            elif w.ndim == 3:
                a, b, c = w.shape
                data[:a, :b, :c] = w
            else:
                raise ValueError("initial core weights must be 1-D vectors or 3-D cores")
            host.append(data)
        cores = [eng.to_device(c) for c in host]
        for i in range(n - 1, 0, -1):
            B, sigma = eng.qr_shift("B", cores[i])
            cores[i] = B
            cores[i - 1] = eng.absorb("B", sigma, cores[i - 1])
        if model.space == "hilbert":
            nrm = math.sqrt(eng.inner(cores[0], cores[0], True).real)
            cores[0] = cores[0] * (scale / nrm)
        else:
            cores[0] = cores[0] * scale
        subspace = {}
        if getattr(model, "subspace_inds", None):
            # Liouville sub-space projection of the finished (right-canonical) MPDO, reference ``project_subspace``
            # (_mps_mpo.py:196-220): keep the listed physical indices, then cut every bond back to the static rule
            # for the reduced site dimensions.  Index selection only -- nothing is re-orthogonalised, as in the reference.
            for isite, P in model.subspace_inds.items():
                P = tuple(int(i) for i in P)
                subspace[int(isite)] = (dims[isite], P)
                idx = torch.as_tensor(P, dtype=torch.long, device=cores[isite].device)
                cores[isite] = cores[isite].index_select(1, idx)
                dims[isite] = len(P)
            for i in range(n):
                ml, mr = bond_dims(dims, i, m)
                cores[i] = cores[i][: (1 if i == 0 else ml), :, : (1 if i == n - 1 else mr)].contiguous()
        me = cls(eng, cores)
        me.subspace = subspace
        return me

    @property
    def sites(self) -> list[SiteCoef]:
        return self.superblock_states[0]

    def bonddim(self) -> list[int]:
        return [s.shape[2] for s in self.sites[:-1]]

    # -- environments --------------------------------------------------------------------------
    @staticmethod
    def construct_op_zerosite() -> dict:
        return {"ovlp": Block(None, True, 1)}

    def renormalize_op_psite(self, psite: int, blocks: dict, H: DeviceMPO, A_is_sys: bool, site: SiteCoef | None = None) -> dict:
        eng = self.eng
        site = self.sites[psite] if site is None else site
        gauge = "A" if A_is_sys else "B"
        t = site.data
        nxt: dict = {}
        ov: Block = blocks["ovlp"]
        if ov.is_identity:
            nxt["ovlp"] = Block(None, True, t.shape[2] if A_is_sys else t.shape[0])
            E_ovlp = None
        else:
            nxt["ovlp"] = Block(eng.env_update(gauge, t, t, ov.data, None), False)
            E_ovlp = ov.data
        for term in H.calc_point[psite + self.site_offset]:
            if (term.is_left and A_is_sys) or (term.is_right and not A_is_sys):
                E = E_ovlp
            else:
                E = blocks[term.key]
            if (term.is_right and A_is_sys) or (term.is_left and not A_is_sys):
                if "summed" in nxt:
                    eng.env_update(gauge, t, t, E, term.core, out=nxt["summed"], accumulate=True)
                else:
                    nxt["summed"] = eng.env_update(gauge, t, t, E, term.core)
            else:
                nxt[term.key] = eng.env_update(gauge, t, t, E, term.core)
        if "summed" in blocks:
            if "summed" in nxt:
                eng.env_update(gauge, t, t, blocks["summed"], None, out=nxt["summed"], accumulate=True)
            else:
                nxt["summed"] = eng.env_update(gauge, t, t, blocks["summed"], None)
        return nxt

    def construct_op_sites(self, begin_site: int, end_site: int, H: DeviceMPO, op_initial_block: dict | None = None,
                           superblock: list | None = None) -> list:
        left = begin_site < end_site
        blocks = [self.construct_op_zerosite() if op_initial_block is None else op_initial_block]
        for p in range(begin_site, end_site, 1 if left else -1):
            blocks.append(self.renormalize_op_psite(p, blocks[-1], H, left, None if superblock is None else superblock[p]))
        return blocks

    @staticmethod
    def _ovlp(blocks) -> torch.Tensor | None:
        ov = blocks["ovlp"]
        return None if ov.is_identity else ov.data

    def operators_for_superH(self, psite: int, op_sys: dict, op_env: dict, H: DeviceMPO, A_is_sys: bool) -> list:
        Lb, Rb = (op_sys, op_env) if A_is_sys else (op_env, op_sys)
        Lo, Ro = self._ovlp(Lb), self._ovlp(Rb)
        terms = []
        if H.coupleJ != 0.0:
            terms.append((Lo, None, Ro, H.coupleJ))
        if "summed" in Lb:
            terms.append((Lb["summed"], None, Ro, 1.0))
        if "summed" in Rb:
            terms.append((Lo, None, Rb["summed"], 1.0))
        for term in H.calc_point[psite + self.site_offset]:
            core = term.core
            # the identity-channel promise holds only while the overlap blocks themselves are identities (canonical MPS)
            if (core.l_id >= 0 and Lo is not None) or (core.r_id >= 0 and Ro is not None):
                core = dataclasses.replace(core, l_id=core.l_id if Lo is None else -1, r_id=core.r_id if Ro is None else -1)
            terms.append((Lb.get(term.key, Lo), core, Rb.get(term.key, Ro), 1.0))
        return terms

    def operators_for_superK(self, op_sys: dict, op_env: dict, H: DeviceMPO, A_is_sys: bool, bond: int | None = None) -> list:
        """``bond`` = local index b of the bond between sites b-1 and b (enables the identity-channel shortcut)."""
        Lb, Rb = (op_sys, op_env) if A_is_sys else (op_env, op_sys)
        Lo, Ro = self._ovlp(Lb), self._ovlp(Rb)
        terms = []
        if H.coupleJ != 0.0:
            terms.append((Lo, Ro, H.coupleJ))
        if "summed" in Lb:
            terms.append((Lb["summed"], Ro, 1.0))
        if "summed" in Rb:
            terms.append((Lo, Rb["summed"], 1.0))
        for key in op_sys.keys():
            if key in ("summed", "ovlp"):
                continue
            assert key in Lb and key in Rb, f"key {key} should be included in summed"
            ids = None
            if bond is not None and Lo is None and Ro is None:
                ids = getattr(H, "bond_ids", {}).get((key, bond + self.site_offset))
            terms.append((Lb[key], Rb[key], 1.0, ids))
        return terms

    # -- local exponentials ----------------------------------------------------------------------
    def _n_warmup(self, size: int, site: int) -> int:
        return min(size, min(max(0, self.niter_krylov.get(site, 0) - 2), 15))

    def _expm(self, cfg, sign: complex, dt: float, x: torch.Tensor, site: int, kind: int, shape_out=None, **terms) -> torch.Tensor:
        """``shape_out`` (adaptive bond growth): the tensor is zero-extended to that shape before the solve and the
        blocks of ``hterms`` are padded to square, which is the reference's stack(extend) / split(truncate) operator."""
        size_override = None
        if shape_out is not None and tuple(shape_out) != tuple(x.shape):
            from ._adaptive import _square_terms_h, pad_to

            size_override = x.numel()
            terms = dict(terms, hterms=_square_terms_h(terms["hterms"], shape_out[0], shape_out[2]))
            x = pad_to(x, tuple(shape_out))
        if cfg.relax == "improved":
            # improved relaxation: eigenvector of H_eff per site, the bond (K) step is skipped (_mps_cls.py:1078-1084, 1159-1160)
            if kind == 1:
                return x
            y = x.clone()
            niter = self.eng.lanczos_eigvec(y, terms["hterms"], root=0, thresh=1.0e-09)
            self.niter_krylov[site] = niter
            if self.record_trace:
                self.trace.append((kind, site, niter))
            return y
        n_warm = self._n_warmup(x.numel() if size_override is None else size_override, site)
        y = x.clone()
        if size_override is not None:
            terms = dict(terms, size_override=size_override)
        if cfg.relax:
            # imaginary time: exp(-H dt/2) on sites, exp(+K dt/2) on bonds, always the Lanczos variant (_mps_cls.py:1086-1094)
            scale = (sign * -1j).real * (dt / 2)
            niter = self.eng.krylov_expm("lanczos", scale, cfg.thresh_exp, n_warm, cfg.conserve_norm, y, **terms)
        else:
            niter = self.eng.krylov_expm(cfg.integrator, sign * (dt / 2), cfg.thresh_exp, n_warm, cfg.conserve_norm, y, **terms)
        self.niter_krylov[site] = niter
        if self.record_trace:
            self.trace.append((kind, site, niter))
        return y

    # -- sweeps ------------------------------------------------------------------------------------
    def propagate_along_sweep(self, H: DeviceMPO, dt: float, cfg, *, begin_site: int, end_site: int,
                              op_sys_initial: dict | None = None, skip_end_site: bool = False) -> dict:
        eng = self.eng
        A_is_sys = begin_site <= end_site
        step = 1 if A_is_sys else -1
        to = "->" if A_is_sys else "<-"
        sites = self.sites
        op_sys = self.construct_op_zerosite() if op_sys_initial is None else op_sys_initial
        if self.op_sys_sites is None:
            env_sites = self.construct_op_sites(end_site, begin_site, H)
        else:
            env_sites = self.op_sys_sites[:]
        self.op_sys_sites = [op_sys]
        adaptive = bool(getattr(cfg, "adaptive", False))
        if adaptive:
            from . import _adaptive as ad

            full = ad.get_superblock_full(eng, sites, cfg.dD)      # neighbours with up to dD complement directions
        for p in range(begin_site, end_site + step, step):
            if skip_end_site and p == end_site:
                return op_sys   # before site_now is touched, as in the reference (_mps_cls.py:878-880)
            self.site_now = p
            op_env = env_sites.pop()
            shape_out = None
            grown = False
            if adaptive and p != end_site:
                L, C, R = sites[p].shape
                if A_is_sys:
                    R = sites[p + 1].shape[0]
                else:
                    L = sites[p - 1].shape[2]
                if not ad.is_max_rank(sites[p], to, cfg.Dmax):
                    grown = True
                    newD, _err, op_env, op_env_braket = ad.get_adaptive_rank_and_block(self, p, full, env_sites[-1], H, to, cfg)
                    if A_is_sys:
                        R = newD
                    else:
                        L = newD
                shape_out = (L, C, R)
            hterms = self.operators_for_superH(p, op_sys, op_env, H, A_is_sys)
            psi = self._expm(cfg, -1.0j, dt, sites[p].data, p, 0, shape_out=shape_out, hterms=hterms)
            sites[p] = SiteCoef(psi, "Psi", p)
            if p == end_site:
                break
            gauge = "A" if A_is_sys else "B"
            new_site, sigma = eng.qr_shift(gauge, psi)
            sites[p] = SiteCoef(new_site, gauge, p)
            op_sys = self.renormalize_op_psite(p, op_sys, H, A_is_sys)
            if grown:
                op_env = op_env_braket
            kterms = self.operators_for_superK(op_sys, op_env, H, A_is_sys, bond=p + 1 if A_is_sys else p)
            sigma = self._expm(cfg, +1.0j, dt, sigma, p, 1, kterms=kterms)
            q = p + step
            sites[q] = SiteCoef(eng.absorb(gauge, sigma, sites[q].data), "Psi", q)
            self.op_sys_sites.append(op_sys)
        return op_sys

    def propagate(self, stepsize: float, H: DeviceMPO, cfg, one_gate: DeviceMPO | None = None, kraus_op: dict | None = None):
        """One time step: forward and backward half sweeps (the last site gets two consecutive half steps); one-site
        gates and Kraus maps, if any, act between the two (reference ``_mps_cls.py:452-503``)."""
        n = self.nsite
        if getattr(cfg, "two_site", False):
            if one_gate is not None or kraus_op is not None:
                raise NotImplementedError("two-site TDVP applies no gates or Kraus maps between its half sweeps")
            from ._twosite import propagate_two_site

            propagate_two_site(self, stepsize, H, cfg)
            return
        self.propagate_along_sweep(H, stepsize, cfg, begin_site=0, end_site=n - 1)
        if one_gate is not None:
            self.apply_one_gate(one_gate, reorth_center=n - 1)
        if kraus_op is not None:
            self.apply_kraus(kraus_op, reorth_center=n - 1)
        self.propagate_along_sweep(H, stepsize, cfg, begin_site=n - 1, end_site=0)

    # -- operator application |Psi'> = O|Psi> / |O|Psi>| (Simulator.operate) ------------------------------------------
    def clone(self) -> "MPSCoefCuda":
        twin = MPSCoefCuda(self.eng, [s.data.clone() for s in self.sites], [s.gauge for s in self.sites])
        twin.subspace = dict(self.subspace)
        return twin

    def apply_dipole(self, init: "MPSCoefCuda", O: DeviceMPO) -> float:
        """One fitting iteration of ``O |init>`` (reference ``MPSCoef.apply_dipole``, _mps_cls.py:421-450): a forward and a
        backward sweep in which every site tensor of THIS chain is replaced by the H_eff-type contraction of ``O`` between this
        chain (bra environments) and ``init`` (ket environments and ket site), normalised; returns the norm found at the last
        site, which converges to |O|init>|.  Both chains are gauge-shifted along the sweep, as in the reference."""
        n = self.nsite
        self._apply_dipole_along_sweep(init, O, 0, n - 1)
        return self._apply_dipole_along_sweep(init, O, n - 1, 0)

    def _apply_dipole_along_sweep(self, init: "MPSCoefCuda", O: DeviceMPO, begin_site: int, end_site: int) -> float:
        """Reference ``apply_dipole_along_sweep`` + ``apply_superOp_direct`` (_mps_cls.py:718-796, 2733-2778).  Environment blocks
        with different bra / ket tensors go through ``tdvp_env_update`` as in the adaptive mode (``_adaptive.renormalize_braket``);
        the site update is one ``tdvp_heff_apply``."""
        from ._adaptive import renormalize_braket

        eng = self.eng
        A_is_sys = begin_site < end_site or self.nsite == 1
        step = 1 if A_is_sys else -1
        bra, ket = self.sites, init.sites
        op_sys = self.construct_op_zerosite()
        cached = getattr(self, "op_sys_sites_dipo", None)
        if cached is None:
            env_sites = [self.construct_op_zerosite()]
            for p in range(end_site, begin_site, -step):
                env_sites.append(renormalize_braket(self, p, env_sites[-1], O, not A_is_sys, bra[p], ket[p]))
        else:
            env_sites = cached[:]
        self.op_sys_sites_dipo = [op_sys]
        norm = 0.0
        gauge = "A" if A_is_sys else "B"
        for p in range(begin_site, end_site + step, step):
            op_env = env_sites.pop()
            hterms = self.operators_for_superH(p, op_sys, op_env, O, A_is_sys)
            new = eng.heff_apply(hterms, ket[p].data)
            norm = math.sqrt(eng.inner(new, new, True).real)
            bra[p] = SiteCoef((new / norm).contiguous(), "Psi", p)
            if p == end_site:
                break
            q = p + step
            for chain in (bra, ket):                     # ..Psi(p) B(p+1).. -> ..A(p) Psi(p+1)..  on both chains
                iso, sigma = eng.qr_shift(gauge, chain[p].data)
                chain[p] = SiteCoef(iso, gauge, p)
                chain[q] = SiteCoef(eng.absorb(gauge, sigma, chain[q].data), "Psi", q)
            op_sys = renormalize_braket(self, p, op_sys, O, A_is_sys, bra[p], ket[p])
            self.op_sys_sites_dipo.append(op_sys)
        return norm

    def apply_kraus(self, kraus_op: dict, reorth_center: int):
        """Kraus maps on a purified MPS (reference ``apply_kraus`` + ``kraus_contract_single_site / _two_site``,
        _mps_cls.py:2375-2418, kraus.py:146-355).  One-site key: the site's physical index is (system d) x (ancilla K);
        two-site key: system site followed by its ancilla site.  The k Kraus operators B[k, x, d] act on the system
        part, the (k, K) pair is compressed back to K ancilla states by an SVD of the (m n x) x (k K) matrix (U S of the K
        largest singular values); the two-site form splits the pair again with a second SVD.  GEMMs + thin SVDs on the device."""
        eng = self.eng
        sb = self.sites
        lo, hi = 10**9, 0
        for site_inds, B in kraus_op.items():
            Bd = B if isinstance(B, torch.Tensor) else eng.to_device(np.asarray(B, dtype=np.complex128))
            k, x, d = Bd.shape
            if len(site_inds) == 1:
                isite = int(site_inds[0])
                lo, hi = min(lo, isite), max(hi, isite)
                A = sb[isite].data
                m, dK, n = A.shape
                if x != d or dK % d:
                    raise ValueError(f"Kraus contract: dK={dK} must be divisible by d={d}")
                K = dK // d
                T = A.reshape(m, d, K * n)
            elif len(site_inds) == 2:
                # system site (d) followed by its ancilla site (K): contract the pair first (kraus.py:258-355)
                i1, i2 = int(site_inds[0]), int(site_inds[1])
                if i1 + 1 != i2:
                    raise ValueError(f"site_inds={site_inds} is not nearest neighbour")
                lo, hi = min(lo, i1), max(hi, i2)
                A1, A2 = sb[i1].data, sb[i2].data
                m, d1, bond = A1.shape
                _, K, n = A2.shape
                if x != d or d1 != d:
                    raise ValueError("Kraus contract: operator and system site dimensions differ")
                T = eng.zgemm(A1.reshape(m * d, bond), A2.reshape(bond, K * n)).reshape(m, d, K * n)
            else:
                raise ValueError(f"site_inds={site_inds} is not yet implemented")
            if m * n * x < K:
                raise ValueError("Kraus contract: fewer rows than ancilla states")
            T2 = T.permute(1, 0, 2).reshape(d, m * K * n).contiguous()                              # [d, (m, K, n)]
            G = eng.zgemm(Bd.reshape(k * x, d).contiguous(), T2).reshape(k, x, m, K, n)              # [k, x, m, K, n]
            if len(site_inds) == 1:
                Cm = G.permute(2, 4, 1, 0, 3).reshape(m * n * x, k * K).contiguous()                 # rows (m, n, x)
                U, sv, _ = eng.svd(Cm)
                scale = torch.as_tensor(sv[:K], dtype=torch.float64, device=U.device)
                sb[isite].data = (U[:, :K] * scale[None, :]).reshape(m, n, x * K).permute(0, 2, 1).contiguous()   # (m, x K, n)
            else:
                Cm = G.permute(2, 1, 4, 0, 3).reshape(m * x * n, k * K).contiguous()                 # rows (m, x, n)
                U, sv, _ = eng.svd(Cm)
                scale = torch.as_tensor(sv[:K], dtype=torch.float64, device=U.device)
                C2 = (U[:, :K] * scale[None, :]).reshape(m, x, n, K).permute(0, 1, 3, 2).reshape(m * x, K * n).contiguous()
                U2, s2, Vh2 = eng.svd(C2)                                                             # split the pair again
                if len(s2) < bond:
                    raise ValueError("Kraus contract: the pair matrix has fewer singular values than the bond dimension")
                sc2 = torch.as_tensor(s2[:bond], dtype=torch.float64, device=U2.device)
                sb[i1].data = (U2[:, :bond] * sc2[None, :]).reshape(m, x, bond).contiguous()
                sb[i2].data = Vh2[:bond, :].reshape(bond, K, n).contiguous()
        canonicalizeB(eng, sb[reorth_center: hi + 1])
        canonicalizeA(eng, sb[lo: reorth_center + 1])
        self.op_sys_sites = None

    def apply_one_gate(self, gate: DeviceMPO, reorth_center: int):
        """U_p on the physical leg of every site that has a gate core, then re-canonicalise around ``reorth_center`` and
        drop the cached environments (reference ``apply_one_gate`` / ``_apply_one_gate_isite``, _mps_cls.py:2314-2451).
        The contraction new[a,i,c] = sum_j U[i,j] old[a,j,c] is stage 2 of the H_eff chain with a (1, d, d, 1) core."""
        sb = self.sites
        changed = []
        for isite in range(self.nsite):
            terms = gate.calc_point[isite + self.site_offset]
            if not terms:
                continue
            if len(terms) >= 2:
                raise ValueError("Multiple one gate on same site is not supported. Contract gates in advance!")
            core = terms[0].core
            if core.wl != 1 or core.wr != 1:
                raise ValueError("one-site gates must be (1, d, d, 1) or (1, d, 1) cores")
            sb[isite].data = self.eng.heff_apply([(None, core, None, 1.0)], sb[isite].data)
            if sb[isite].gauge != "Psi":
                sb[isite].gauge = "C"
                changed.append(isite)
        if changed:
            canonicalizeB(self.eng, sb[reorth_center: max(changed) + 1])
            canonicalizeA(self.eng, sb[min(changed): reorth_center + 1])
            self.op_sys_sites = None

    def hermitise(self):
        """rho <- (rho + rho^dagger) / 2 of a Liouville-space MPDO, compressed back to the bond dimensions it had (reference
        ``MPSCoef.hermitise`` / ``svd_conj_mpdo``, _mps_cls.py:2289-2312, 2516-2562; the reference leaves its call inside
        ``propagate`` commented out, :501-503, so this is an explicit user call here as well).  The sum is the direct-sum
        MPDO [rho/2 | rho^dagger/2] (first site: along the right bond; inner sites: block diagonal; last site: along the
        left bond) with doubled bonds; a left-to-right pass of two-site SVDs truncates every bond back to its original
        dimension (U to the left, S Vh to the right), then the chain is re-canonicalised with the centre on site 0.  One GEMM and
        one thin Jacobi SVD per bond, on the device; the cached environments are dropped."""
        if self.subspace:
            raise NotImplementedError("hermitise: sub-space sites have no square physical index (the reference asserts the same)")
        eng, sb, n = self.eng, self.sites, self.nsite

        def four(t):
            Dl, dd, Dr = t.shape
            q = math.isqrt(dd)
            if q * q != dd:
                raise ValueError("hermitise: Liouville-space sites need a square physical dimension")
            return t.reshape(Dl, q, q, Dr)

        if n == 1:
            rho = four(sb[0].data)
            sb[0].data = (0.5 * (rho + rho.conj().permute(0, 2, 1, 3))).reshape(sb[0].data.shape).contiguous()
            return
        bonds = [int(s.data.shape[-1]) for s in sb[:-1]]
        for i, s in enumerate(sb):
            rho = four(s.data)
            dag = rho.conj().permute(0, 2, 1, 3)
            a, q, _, d = rho.shape
            if i == 0:
                data = torch.cat((0.5 * rho, 0.5 * dag), dim=3)
            elif i == n - 1:
                data = torch.cat((rho, dag), dim=0)
            else:
                data = torch.zeros((2 * a, q, q, 2 * d), dtype=rho.dtype, device=rho.device)
                data[:a, :, :, :d] = rho
                data[a:, :, :, d:] = dag
            s.data = data.reshape(data.shape[0], q * q, data.shape[3]).contiguous()
        for i in range(n - 1):
            L, R = sb[i].data, sb[i + 1].data
            a, j, k = L.shape
            _, l, m = R.shape
            chi = bonds[i]
            if chi > min(a * j, l * m):
                raise ValueError("hermitise: bond dimension exceeds the rank of the two-site matrix")
            two = eng.zgemm(L.reshape(a * j, k).contiguous(), R.reshape(k, l * m).contiguous())
            U, sv, Vh = eng.svd(two)
            scale = torch.as_tensor(np.asarray(sv[:chi]), dtype=torch.float64, device=U.device)
            sb[i].data = U[:, :chi].contiguous().reshape(a, j, chi)
            sb[i + 1].data = (scale[:, None] * Vh[:chi, :]).contiguous().reshape(chi, l, m)
        canonicalize(eng, sb, 0, incremental=False)
        self.op_sys_sites = None

    # -- observables ---------------------------------------------------------------------------------
    def _liouville_four(self, isite: int) -> torch.Tensor:
        """Site tensor of an MPDO as (D_l, q, q, D_r); sub-space sites are embedded back into the full q x q index first
        (reference ``define_reshape_mat`` / ``_reshape_core``, _mps_mpo.py:135-194)."""
        t = self.sites[isite].data
        Dl, dd, Dr = t.shape
        if isite + self.site_offset in self.subspace:
            full_d, P = self.subspace[isite + self.site_offset]
            full = torch.zeros((Dl, full_d, Dr), dtype=t.dtype, device=t.device)
            full[:, torch.as_tensor(P, dtype=torch.long, device=t.device), :] = t
            t, dd = full, full_d
        q = math.isqrt(dd)
        if q * q != dd:
            raise ValueError("Liouville-space sites need a square physical dimension")
        return t.reshape(Dl, q, q, Dr)

    def _exp_liouville(self, H: DeviceMPO) -> complex:
        """Tr(O rho) of a Liouville-space MPDO for a Hilbert-space operator O given as MPO cores of physical dimension
        q = sqrt(d) (reference ``_exp_liouville``, _mps_cls.py:3769-3838: per MPO key a left-to-right chain
        "ab,bcde,adcf->fe"; sites the key does not touch contribute their partial trace "ab,bcce->ae").  Two DMMA GEMMs
        per site and key; no canonical form is needed.  As in the reference the scalar ``coupleJ`` term is not included."""
        eng = self.eng
        by_key: dict = {}
        for p, terms in enumerate(H.calc_point):
            for t in terms:
                by_key.setdefault(t.key, {})[p] = t.core
        total = 0.0 + 0.0j
        four = [self._liouville_four(i) for i in range(self.nsite)]
        for key, cores in by_key.items():
            left = torch.ones((1, 1), dtype=torch.complex128, device=eng.torch_device)
            for isite in range(self.nsite):
                t4 = four[isite]
                Dl, q, _, Dr = t4.shape
                core = cores.get(isite + self.site_offset)
                if core is None:
                    m = torch.diagonal(t4, dim1=1, dim2=2).sum(-1).contiguous()              # partial trace: (D_l, D_r)
                    left = eng.zgemm(left, m)
                    continue
                w = int(left.shape[0])
                if core.wl != w or int(core.data.shape[1]) != q:
                    raise ValueError(f"observable core at site {isite} has shape {tuple(core.data.shape)}; expected MPO bond {w} "
                                     f"and the Hilbert-space dimension {q} of a Liouville site of dimension {q * q}")
                X = eng.zgemm(left, t4.reshape(Dl, q * q * Dr).contiguous())                 # [a, (c, d, e)]
                if core.data.dim() == 4:
                    perm = core.perm if core.perm is not None else core.data.permute(0, 2, 1, 3).contiguous()
                    Wm = perm.reshape(w * q * q, core.wr)                                     # perm[a, c, d, f] = W[a, d, c, f]
                    left = eng.zgemm(Wm, X.reshape(w * q * q, Dr), transA=1)
                else:                                                                          # diagonal core W[a, c, f]
                    Xd = torch.diagonal(X.reshape(w, q, q, Dr), dim1=1, dim2=2).permute(0, 2, 1).contiguous()
                    left = eng.zgemm(core.data.reshape(w * q, core.wr), Xd.reshape(w * q, Dr), transA=1)
            if tuple(left.shape) != (1, 1):
                raise ValueError(f"MPO key {key} does not close: final block has shape {tuple(left.shape)}")
            total += complex(left.cpu().numpy()[0, 0])
        return total

    def expectation(self, H: DeviceMPO, space: str = "hilbert") -> complex:
        """<Psi|Op|Psi> at the centre site 0: full right-environment rebuild + one matvec + inner product.
        ``space="liouville"``: Tr(Op rho) of the vectorised density matrix instead (``_exp_liouville``)."""
        if space == "liouville":
            return self._exp_liouville(H)
        assert self.sites[0].gauge == "Psi", "the MPS must be canonical around site 0"
        n = self.nsite
        env = self.construct_op_sites(n - 1, 0, H).pop() if n > 1 else self.construct_op_zerosite()
        terms = self.operators_for_superH(0, self.construct_op_zerosite(), env, H, True)
        psi = self.sites[0].data
        return self.eng.inner(psi, self.eng.heff_apply(terms, psi), True)

    def autocorr(self) -> complex:
        """<Psi(t/2)^*|Psi(t/2)> (t/2 trick) as a chain of overlap-site contractions."""
        return self._overlap(conj=False)

    def _overlap(self, conj: bool) -> complex:
        eng = self.eng
        block = torch.ones((1, 1), dtype=torch.complex128, device=eng.torch_device)
        for s in self.sites:
            block = eng.overlap_site(s.data, s.data, block, conj)
        return complex(block.cpu().numpy()[0, 0])

    def pop_states(self) -> list[float]:
        psi = self.sites[0].data
        return [self.eng.inner(psi, psi, True).real]

    def norm(self) -> float:
        return math.sqrt(sum(self.pop_states()))

    # -- reduced densities (SURVEY 8(f1); reference _mps_cls.py:1208-1287, 1628-1678) ---------------------
    def _pure_reduced_density(self, remain_nleg: tuple[int, ...]) -> np.ndarray:
        """rho of the sites flagged in ``remain_nleg`` (0 = traced, 1 = diagonal only, 2 = ket and bra legs); index
        order = site order, ket before bra.  Contracted right to left over the first len(remain_nleg) sites; the B-gauge
        sites further right drop out.  Both contractions per site are DMMA GEMMs; index shuffles are strided copies."""
        eng = self.eng
        if self.sites[0].gauge != "Psi" or any(s.gauge != "B" for s in self.sites[1:]):
            raise ValueError("the MPS must be canonical around site 0")
        if len(remain_nleg) > self.nsite or not remain_nleg or remain_nleg[-1] not in (1, 2) or any(
                n not in (0, 1, 2) for n in remain_nleg):
            raise ValueError(f"invalid remain_nleg {remain_nleg}: entries 0/1/2, the last one 1 or 2")
        cores = [s.data for s in self.sites[: len(remain_nleg)]]
        C = cores.pop()
        i, j, k = C.shape
        Cm = C.reshape(i * j, k)
        dens = eng.zgemm(Cm, Cm, 0, 2).reshape(i, j, i, j).permute(0, 2, 1, 3)   # [i, a, ket j, bra l]
        if remain_nleg[-1] == 1:
            dens = torch.diagonal(dens, dim1=2, dim2=3)
        dens = dens.contiguous()
        isite = len(remain_nleg) - 1
        while cores:
            isite -= 1
            nleg = remain_nleg[isite]
            C = cores.pop()
            l, m, i = C.shape
            a = dens.shape[1]
            xshape = tuple(dens.shape[2:])
            x = int(np.prod(xshape)) if xshape else 1
            T = eng.zgemm(C.reshape(l * m, i), dens.reshape(i, a * x)).reshape(l, m, a, x)      # [l, m, a, X]
            if nleg == 0:
                T2 = T.permute(0, 3, 1, 2).reshape(l * x, m * a).contiguous()                  # [(l, X), (m, a)]
                new = eng.zgemm(T2, C.reshape(l, m * a), 0, 2).reshape(l, x, l).permute(0, 2, 1)  # [l, b, X]
                dens = new.reshape((l, l) + xshape).contiguous()
            else:
                T2 = T.permute(0, 1, 3, 2).reshape(l * m * x, a).contiguous()                  # [(l, m, X), a]
                new = eng.zgemm(T2, C.reshape(l * m, a), 0, 2).reshape(l, m, x, l, m)          # [l, m, X, b, n]
                new = new.permute(0, 3, 1, 4, 2)                                               # [l, b, m, n, X]
                if nleg == 1:
                    new = torch.diagonal(new, dim1=2, dim2=3).permute(0, 1, 3, 2)              # [l, b, m, X]
                    dens = new.reshape((l, l, m) + xshape).contiguous()
                else:
                    dens = new.reshape((l, l, m, m) + xshape).contiguous()
        return dens[0, 0].cpu().numpy()

    def _partial_trace(self, remain_nleg: tuple[int, ...]) -> np.ndarray:
        """Liouville-space MPDO (physical index = vectorised d x d matrix): partial trace keeping the flagged sites
        (reference ``get_partial_trace``, _mps_cls.py:1438-1510; no canonical form needed).  Traced sites contribute the
        D x D transfer matrix sum_j core[:, (j, j), :]; everything is O(n D^2 d^2) index work on the device tensors."""
        center = max((i for i, n in enumerate(remain_nleg) if n in (1, 2)), default=None)
        if center is None:
            raise ValueError("No site with 2 legs found in remain_nleg")
        four = [self._liouville_four(i) for i in range(self.nsite)]
        left = torch.ones(1, dtype=torch.complex128, device=four[0].device)
        for isite in range(center):
            t = four[isite]
            if remain_nleg[isite] == 0:
                m = torch.diagonal(t, dim1=1, dim2=2).sum(-1)                          # ijjl -> il
            elif remain_nleg[isite] == 1:
                m = torch.diagonal(t, dim1=1, dim2=2).permute(0, 2, 1)                 # ijjl -> ijl
            elif remain_nleg[isite] == 2:
                m = t
            else:
                raise ValueError(f"Invalid number of legs: {remain_nleg[isite]}")
            left = torch.tensordot(left, m, dims=([left.dim() - 1], [0]))
        right = torch.ones(1, dtype=torch.complex128, device=four[0].device)
        for isite in range(self.nsite - 1, center, -1):
            right = torch.diagonal(four[isite], dim1=1, dim2=2).sum(-1) @ right
        dm = torch.tensordot(left, torch.tensordot(four[center], right, dims=([3], [0])), dims=([left.dim() - 1], [0]))
        return dm.cpu().numpy()

    def get_reduced_densities(self, remain_nleg, space: str = "hilbert") -> list[np.ndarray]:
        """Reference ``MPSCoef.get_reduced_densities``: one key (tuple) or a list of keys -> list of arrays; pure-state
        reduced densities in Hilbert space, partial traces of the MPDO in Liouville space."""
        if isinstance(remain_nleg, tuple):
            remain_nleg = [remain_nleg]
        if space == "liouville":
            return [self._partial_trace(tuple(k)) for k in remain_nleg]
        return [self._pure_reduced_density(tuple(k)) for k in remain_nleg]

    def to_numpy(self) -> list[np.ndarray]:
        return [s.numpy() for s in self.sites]
