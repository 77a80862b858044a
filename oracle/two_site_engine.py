"""``OracleEngine`` with the two-site calls of ``pytdscf_b200._engine.Engine`` (``heff2_apply``, ``krylov_expm2``,
``split2``) on the NumPy kernels of ``oracle/two_site_oracle.py`` -- TEST INFRASTRUCTURE.  The same strict contract checks as
the one-site methods: contiguous complex128 tensors, consistent shapes, a promised identity channel verified numerically."""
from __future__ import annotations

import numpy as np

from oracle import tdvp_oracle as orc
from oracle import two_site_oracle as tso
from oracle.oracle_engine import OracleEngine, _chk, _chk_shortcut, _core, _np, _unit_channel


class TwoSiteOracleEngine(OracleEngine):
    # -- two-site TDVP -----------------------------------------------------------------------------------------------
    def _chk_h2terms(self, terms, theta):
        Dl, d1, d2, Dr = theta.shape
        for L, c1, c2, R, _coef in terms:
            _chk(L, "L", 3)
            _chk(R, "R", 3)
            if L is not None and (L.shape[0] != Dl or L.shape[2] != Dl) or R is not None and (R.shape[0] != Dr or R.shape[2] != Dr):
                raise ValueError(f"two-site block does not match theta {tuple(theta.shape)}")
            c1 = None if c1 is None or c1.data is None else c1
            c2 = None if c2 is None or c2.data is None else c2
            wl = 1 if L is None else L.shape[1]
            wr = 1 if R is None else R.shape[1]
            wm = c1.wr if c1 is not None else (c2.wl if c2 is not None else 1)
            for c, d, a, b in ((c1, d1, wl, wm), (c2, d2, wm, wr)):
                if c is None:
                    if a != 1 or b != 1:
                        raise ValueError("an identity core needs MPO bond dimensions of 1 on both of its sides")
                    continue
                _chk(c.data, "W")
                if c.data.shape[1] != d:
                    raise ValueError("core / site physical dimension mismatch")
                if c.wl != a or c.wr != b:
                    raise ValueError("two-site term: block / core bond dimensions do not match")

    @staticmethod
    def _heff2_sum(terms, theta) -> np.ndarray:
        return tso.heff2_apply([(_np(L), _core(c1), _core(c2), _np(R), coef) for L, c1, c2, R, coef in terms], theta.numpy())

    def heff2_apply(self, terms, theta):
        if self.strict:
            _chk(theta, "theta", 4)
            self._chk_h2terms(terms, theta)
        out = self._heff2_sum(terms, theta)
        if self.strict:
            promised = [(L, c1, c2, R, coef) for (L, c1, c2, R, coef) in terms
                        if (L is not None and c1 is not None and c1.data is not None and c1.l_id >= 0)
                        or (R is not None and c2 is not None and c2.data is not None and c2.r_id >= 0)]
            if promised:
                def unit(B, c, side):
                    ch = None if c is None or c.data is None else (c.l_id if side == "l" else c.r_id)
                    return B if B is None or ch is None or ch < 0 else _unit_channel(B, ch)

                short = [(unit(L, c1, "l"), c1, c2, unit(R, c2, "r"), coef) for (L, c1, c2, R, coef) in promised]
                _chk_shortcut(self._heff2_sum(promised, theta), self._heff2_sum(short, theta), "two-site H_eff")
        return self._wrap(out)

    def krylov_expm2(self, kind, scale, thresh, n_warmup, conserve_norm, theta, terms):
        if self.strict:
            _chk(theta, "theta", 4)
            self._chk_h2terms(terms, theta)
        last = n_warmup + 2 if n_warmup > 0 else 0
        mv = lambda x: self.heff2_apply(terms, self._wrap(x)).numpy()  # noqa: E731
        solver = orc.sia_reference if kind == "arnoldi" else orc.sil_reference
        y, n = solver(complex(scale), mv, theta.numpy().copy(), thresh, last_niter=last, conserve_norm=conserve_norm)
        theta.copy_(self._wrap(y))
        self._stats["solves"] += 1
        self._stats["matvecs"] += n
        return n

    def split2(self, direction, theta, p, Dcap, conserve_norm):
        self._pre((theta, "theta", 4))
        self._require(direction in ("left", "right") and 0.0 <= p < 1.0 and Dcap >= 1, "split2: bad argument")
        left, right, s, r = tso.split_two_site(theta.numpy(), direction, p, Dcap, conserve_norm)
        return self._wrap(left), self._wrap(right), s, r
