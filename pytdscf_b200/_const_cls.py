"""Run configuration (reference: the global ``const`` of ``pytdscf/_const_cls.py:102-252``).

Unlike the reference this is an explicit object owned by the ``Simulator`` (no mutable module global), but the
field names and the rules that derive them are the same."""
from __future__ import annotations

from dataclasses import dataclass


@dataclass
class RunConfig:
    jobname: str = "propagate"
    relax: bool | str = False
    maxstep: int = 9999999
    thresh_exp: float = 1.0e-09  # = thresh_sil
    verbose: int = 2
    space: str = "hilbert"
    integrator: str = "lanczos"
    conserve_norm: bool = True
    display_time_unit: str = "fs"
    time_au_init: float = 0.0
    adaptive: bool = False
    Dmax: int = 20       # adaptive_Dmax
    dD: int = 5          # adaptive_dD
    p_proj: float = 1.0e-04  # adaptive_p_proj
    p_svd: float = 1.0e-07  # adaptive_p_svd: truncation weight of the site-parallel boundary bond (reference const.p_svd)
    two_site: bool = False  # two-site TDVP: bonds follow the state (truncated SVD split of every pair)
    two_site_p_svd: float = 1.0e-07  # truncation weight of the two-site split (the rule of adaptive_p_svd)
    bond_dim: int = 0  # two-site TDVP: bond-dimension cap (the model's bond_dim; 0 = matricisation ranks only)

    def __post_init__(self):
        self.space = self.space.lower()
        self.integrator = self.integrator.lower()
        if self.space not in ("hilbert", "liouville"):
            raise ValueError(f"space must be 'hilbert' or 'liouville' but got {self.space}")
        if self.integrator not in ("lanczos", "arnoldi"):
            raise ValueError(f"Invalid integrator: {self.integrator}")
        if self.space == "liouville":  # _const_cls.py:219-224
            self.conserve_norm = False
        if self.adaptive and self.relax:
            raise NotImplementedError("adaptive bond dimensions are implemented for real-time propagation only")
        if self.two_site and (self.relax or self.adaptive):
            raise NotImplementedError("two-site TDVP is implemented for real-time propagation without adaptive=True")
