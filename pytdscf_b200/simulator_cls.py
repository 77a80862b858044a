"""``Simulator``: the user-facing driver with the reference's signature plus ``backend="cuda"``.

Reference: ``pytdscf/simulator_cls.py:34-592`` (constructor :58-75, ``propagate`` :160-284, time loop
``_execute`` :332-467), ``pytdscf/wavefunction.py`` (``WFunc``) and ``pytdscf/properties.py`` (per-step
observables and the ``<jobname>_prop/*.dat`` files).  Differences by design: there is exactly one backend
("cuda", no dispatch, no CPU fallback), the run configuration is an explicit object instead of a mutable
global, and the checkpoint is a plain pickle of NumPy cores instead of a ``dill`` dump of live objects.
"""
from __future__ import annotations

import os
import pickle
import time as _time

import numpy as np

from . import units
from ._const_cls import RunConfig
from ._engine import Engine
from ._mps_cuda import DeviceMPO, MPSCoefCuda
from .model_cls import Model


class WFunc:
    """Wavefunction = device MPS + the operators it is measured against (reference ``wavefunction.py:34-598``)."""

    def __init__(self, ci_coef: MPSCoefCuda, eng: Engine, space: str = "hilbert"):
        self.ci_coef = ci_coef
        self.eng = eng
        self.space = space
        self._dev_ops: dict[int, DeviceMPO] = {}
        self.merge_mpo_terms = False   # set by Simulator: direct-sum the whole-chain MPO keys (launch-bound small-D runs)

    def device_op(self, op) -> DeviceMPO:
        key = id(op)
        if key not in self._dev_ops:
            self._dev_ops[key] = DeviceMPO(self.eng, op, merge_terms=self.merge_mpo_terms)
        return self._dev_ops[key]

    def expectation(self, op) -> float:
        """Real part of <Psi|Op|Psi> (reference ``wavefunction.py:90-114`` also returns ``.real``)."""
        val = self.ci_coef.expectation(self.device_op(op), space=self.space) if self.space == "liouville" else \
            self.ci_coef.expectation(self.device_op(op))
        return None if val is None else val.real   # site-parallel runs: only rank 0 holds the value

    def autocorr(self) -> complex:
        return self.ci_coef.autocorr()

    def norm(self) -> float:
        return self.ci_coef.norm()

    def pop_states(self) -> list[float]:
        return self.ci_coef.pop_states()

    def bonddim(self) -> list[int]:
        return self.ci_coef.bonddim()

    def get_reduced_densities(self, remain_nleg) -> list[np.ndarray]:
        """Reduced density matrices (reference ``wavefunction.py:67-88``); 0 = traced, 1 = diagonal, 2 = both legs."""
        return self.ci_coef.get_reduced_densities(remain_nleg, space=self.space)

    def apply_dipole(self, matOp, maxstep: int = 10, conv_tol: float = 1.0e-08, log=None) -> float:
        """|Psi> <- O|Psi> / |O|Psi>| by fitting sweeps; returns |O|Psi>| (reference ``WFunc.apply_dipole`` / ``_is_converged``,
        wavefunction.py:285-351): at most ``maxstep`` iterations, stopped when the overlap with the previous iterate is 1 to 1e-8."""
        mps = self.ci_coef
        O = self.device_op(matOp)
        init = mps.clone()
        mps.op_sys_sites_dipo = None
        norm = 0.0
        for it in range(maxstep):
            prev = mps.clone()
            norm = mps.apply_dipole(init, O)
            block = None
            for b, k in zip(mps.sites, prev.sites, strict=True):
                if block is None:
                    block = self.eng.to_device(np.ones((1, 1), dtype=np.complex128))
                block = self.eng.overlap_site(b.data, k.data, block, True)
            ovlp = complex(block.cpu().numpy()[0, 0])
            if log is not None:
                log(f"iterations: {it} norm: {norm} convergence: {abs(ovlp)}")
            if abs(1.0 - abs(ovlp)) < conv_tol:
                break
        else:
            if log is not None:
                log(f"Operate O|Psi> is not converged in {maxstep} iterations")
        mps.op_sys_sites = None        # environments of a Hamiltonian, if any were cached, belong to the old state
        return norm

    def propagate_SM(self, matH, stepsize: float, cfg: RunConfig, one_gate_to_apply=None, kraus_op=None):
        if one_gate_to_apply is None and kraus_op is None:
            self.ci_coef.propagate(stepsize, self.device_op(matH), cfg)
        else:
            if kraus_op is not None and getattr(self, "_kraus_dev", None) is None:
                self._kraus_dev = {k: self.eng.to_device(v) for k, v in kraus_op.items()}     # uploaded once
            self.ci_coef.propagate(stepsize, self.device_op(matH), cfg,
                                   one_gate=None if one_gate_to_apply is None else self.device_op(one_gate_to_apply),
                                   kraus_op=None if kraus_op is None else self._kraus_dev)


class _DatFile:
    def __init__(self, path: str):
        self.f = open(path, "w")

    def write(self, line: str):
        self.f.write(line + "\n")
        self.f.flush()

    def close(self):
        self.f.close()


def _write_reduced_density_nc(path: str, rows: list, display_time_unit: str = "fs") -> str | None:
    """``<job>/reduced_density.nc`` with the reference's layout (pytdscf/properties.py:160-213): unlimited dimension ``step``,
    ``state``, one dimension ``Q<site>`` per site of a key, variable ``time`` (display unit) and one variable
    ``rho_<key>_<state>`` per key with dimensions (step, Q.., Q..).  The reference writes NETCDF4 with a compound
    (real, imag) type through the netCDF4 package; neither that package nor HDF5 exists here, so the file is NetCDF-3
    (64-bit offset, written by ``scipy.io.netcdf_file``; the netCDF4 package and xarray read it too) and the complex values carry a
    trailing dimension ``complex`` of length 2 = (real, imag) instead of the compound type.  Skipped when SciPy is missing."""
    try:
        from scipy.io import netcdf_file
    except ImportError:      # pragma: no cover
        return None
    from .units import au_in_fs

    scale = {"fs": au_in_fs, "ps": au_in_fs * 1.0e-3, "au": 1.0}.get(display_time_unit, au_in_fs)
    with netcdf_file(path, "w", version=2) as f:
        f.createDimension("step", None)
        f.createDimension("state", 1)
        f.createDimension("complex", 2)
        t = f.createVariable("time", "d", ("step",))
        t.units = display_time_unit if display_time_unit in ("fs", "ps", "au") else "fs"
        var = {}
        for key, rho in rows[0]["reduced_densities"].items():
            dims = []
            for idof, n in zip(key, np.asarray(rho).shape, strict=True):
                name = f"Q{idof}"
                if name not in f.dimensions:
                    f.createDimension(name, int(n))
                dims.append(name)
            var[key] = f.createVariable(f"rho_{tuple(key)}_0", "d", ("step", *dims, "complex"))
        for i, r in enumerate(rows):
            t[i] = r["time_au"] * scale
            for key, rho in r["reduced_densities"].items():
                rho = np.asarray(rho)
                var[key][i] = np.stack([rho.real, rho.imag], axis=-1)
    return path


class Simulator:
    """The simulator of the PyTDSCF-style API, running on one B200 through libtdvp_b200.

    Args:
        jobname (str): prefix of the output directory ``<jobname>_prop`` and of ``wf_<jobname>.pkl``.
        model (Model): basis + operators.
        ci_type (str): only ``"mps"``.
        backend (str): only ``"cuda"`` -- there is no NumPy/JAX path in this package.
        t2_trick (bool): autocorrelation by <Psi(t/2)*|Psi(t/2)> (the only implemented form).
        verbose (int): 0..4 as in the reference (>= 2 prints per-step lines to main.log).
        device (int | None): CUDA device ordinal (default: torch's current device).
    """

    def __init__(self, jobname: str, model: Model, ci_type: str = "mps", backend: str = "cuda", proj_gs: bool = False,
                 t2_trick: bool = True, verbose: int = 2, device: int | None = None):
        if backend.lower() != "cuda":
            raise ValueError(f"backend must be 'cuda' in pytdscf_b200 (got {backend!r}); there is no NumPy/JAX dispatch")
        if ci_type.lower() != "mps":
            raise ValueError(f"ci_type must be 'mps' (MCTDH / full-CI coefficients are out of scope), got {ci_type}")
        if proj_gs:
            raise NotImplementedError("proj_gs belongs to the SPF layer, which is out of scope")
        if not t2_trick:
            raise NotImplementedError("only the t/2-trick autocorrelation is implemented")
        self.jobname = jobname
        self.model = model
        self.model.apply_backend("cuda")
        self.verbose = verbose
        self.device = device
        self.eng: Engine | None = None
        self.history: list[dict] = []  # full-precision per-step observables (state BEFORE each step)
        self.cfg: RunConfig | None = None

    # -----------------------------------------------------------------------------------------------
    def _engine(self) -> Engine:
        if self.eng is None:
            self.eng = Engine(self.device)
        return self.eng

    def save_wavefunction(self, wf: WFunc, ext: str = "", reference_format: bool = False):
        """``wf_<jobname><ext>.pkl``: NumPy site tensors + gauge labels (own format), or -- ``reference_format=True`` -- a
        pickle that the reference's ``Simulator(...).propagate(restart=True)`` loads as its own ``WFunc``
        (pytdscf/simulator_cls.py:501-507; see ``pytdscf_b200/checkpoint.py``)."""
        path = f"wf_{self.jobname}{ext}.pkl"
        cores, gauges = wf.ci_coef.to_numpy(), [s.gauge for s in wf.ci_coef.sites]
        if reference_format:
            from .checkpoint import write_reference_wavefunction

            return write_reference_wavefunction(path, cores, gauges)
        with open(path, "wb") as f:
            pickle.dump({"cores": cores, "gauges": gauges}, f)
        return path

    def load_wavefunction(self, ext: str = "") -> WFunc:
        """Load ``wf_<jobname><ext>.pkl`` written by this package OR by the reference (a ``dill`` dump of its ``WFunc``,
        pytdscf/simulator_cls.py:577-589; read without importing the reference)."""
        from .checkpoint import is_reference_pickle, read_reference_wavefunction

        path = f"wf_{self.jobname}{ext}.pkl"
        if is_reference_pickle(path):
            d = read_reference_wavefunction(path)
        else:
            with open(path, "rb") as f:
                d = pickle.load(f)
        eng = self._engine()
        return WFunc(MPSCoefCuda.from_user_cores(eng, d["cores"], d["gauges"]), eng, self.model.space)

    def set_initial_mps(self, cores: list, gauges: list[str] | None = None):
        """Lower-level entry: start from explicit site tensors (site 0 = centre, the rest right-canonical)."""
        self._initial_mps = ([np.asarray(c, dtype=np.complex128) for c in cores], gauges)

    def get_initial_wavefunction(self, restart: bool = False, loadfile_ext: str = "") -> WFunc:
        if restart:
            return self.load_wavefunction(loadfile_ext)
        eng = self._engine()
        if getattr(self, "_initial_mps", None) is not None:
            cores, gauges = self._initial_mps
            return WFunc(MPSCoefCuda.from_user_cores(eng, cores, gauges), eng, self.model.space)
        return WFunc(MPSCoefCuda.alloc_random(eng, self.model), eng, self.model.space)

    def _distributed_wavefunction(self, split: list[tuple[int, ...]]) -> WFunc:
        """Site-segment-parallel start: rank 0 canonicalises the serial initial MPS and scatters the segments."""
        from . import parallel
        from ._mps_parallel import Comm, MPSCoefParallelCuda

        info = getattr(self, "rank_info", None) or parallel.init_from_env()
        self.rank_info = info
        if info.world != len(split) or info.world < 2:
            raise ValueError(f"parallel_split_indices has {len(split)} segments but the process group has {info.world} "
                             "ranks (launch with torchrun --nproc-per-node <segments>)")
        n = self.model.get_ndof()
        # the reference reads only the first and last entry of every tuple (_const_cls.py:236-250): (start, end) pairs -- its
        # documented form -- and tuples that list every site of the segment are both accepted
        ok = split[0][0] == 0 and split[-1][-1] == n - 1 and all(seg[0] <= seg[-1] for seg in split)
        ok = ok and all(split[i][-1] + 1 == split[i + 1][0] for i in range(len(split) - 1))
        if not ok:
            raise ValueError("parallel_split_indices must partition 0..nsite-1 into consecutive segments")
        eng = self._engine()
        comm = Comm(info, eng.torch_device)
        # operators built on rank 0 only (the reference's MPI idiom, ``TensorHamiltonian(potential=None)`` elsewhere): rank 0
        # hands its host cores to every rank; nothing is exchanged when every rank built its own
        ham = self.model.hamiltonian
        if comm.allreduce_lor(bool(getattr(ham, "deferred", False))):
            if comm.allreduce_lor(info.rank == 0 and ham.deferred):      # every rank learns it, so nobody is left waiting
                raise ValueError("rank 0 must hold the Hamiltonian (potential=None is for the other ranks)")
            if info.rank == 0:
                payload = ham.export_cores()
                for r in range(1, info.world):
                    comm.send(payload, r)
            else:
                payload = comm.recv(0)
                if ham.deferred:
                    ham.adopt(payload)
        cores = None
        if getattr(self, "_initial_mps", None) is not None:
            cores = self._initial_mps[0]
        mps = MPSCoefParallelCuda.distribute(eng, comm, self.model, [seg[0] for seg in split], cores=cores)
        return WFunc(mps, eng)

    # -----------------------------------------------------------------------------------------------
    def propagate(self, stepsize: float = 0.1, maxstep: int = 5000, restart: bool = False, savefile_ext: str = "",
                  loadfile_ext: str = "_operate", backup_interval: int = 1000, autocorr: bool = True,
                  energy: bool = True, norm: bool = True, populations: bool = True, observables: bool = False,
                  reduced_density=None, Δt: float | None = None, thresh_sil: float = 1.0e-09,
                  autocorr_per_step: int = 1, observables_per_step: int = 1, energy_per_step: int = 1,
                  norm_per_step: int = 1, populations_per_step: int = 1, parallel_split_indices=None,
                  adaptive: bool = False, adaptive_Dmax: int = 20, adaptive_dD: int = 5,
                  adaptive_p_proj: float = 1.0e-04, adaptive_p_svd: float = 1.0e-07, integrator: str = "lanczos",
                  display_time_unit: str = "fs", conserve_norm: bool = True, write_files: bool = True,
                  record_trace: bool = False, two_site: bool = False, two_site_p_svd: float = 1.0e-07):
        """Real-time propagation; returns ``(energy, wf)`` like the reference (energy of the last evaluated step).

        ``two_site=True``: two-site TDVP -- every pair of neighbouring sites is propagated together and split again by a
        truncated SVD, so the bond dimensions follow the state (from a Hartree product up to the model's ``bond_dim``):
        the smallest rank whose cumulative singular-value sum reaches ``1 - two_site_p_svd`` of the total is kept.  Bond
        dimensions are written to ``bonddim.dat`` and ``history``.  Not combined with ``adaptive``, site-parallel runs,
        gates or Kraus maps."""
        if two_site:
            if adaptive:
                raise NotImplementedError("two_site=True and adaptive=True are alternative bond-growth schemes; pick one")
            if parallel_split_indices is not None:
                raise NotImplementedError("two-site TDVP is not implemented for site-parallel runs")
            if self.model.one_gate_to_apply is not None or self.model.kraus_op is not None:
                raise NotImplementedError("two-site TDVP applies no gates or Kraus maps between its half sweeps")
            if self.model.get_ndof() < 2:
                raise ValueError("two-site TDVP needs a chain of at least two sites")
            if not 0.0 <= two_site_p_svd < 1.0:
                raise ValueError(f"two_site_p_svd must lie in [0, 1), got {two_site_p_svd}")
        self._two_site = (bool(two_site), float(two_site_p_svd))
        self._rd = None
        if reduced_density is not None:
            keys, rd_step = reduced_density
            legs = []
            for key in keys:   # site indices -> legs per site, as properties.py:64-83: (0, 0) -> (2,), (1, 2) -> (0, 1, 1)
                cnt = [0] * (max(key) + 1)
                for isite in key:
                    cnt[isite] += 1
                if any(c > 2 for c in cnt):
                    raise ValueError(f"reduced_density key {key}: a site may appear at most twice")
                legs.append(tuple(cnt))
            self._rd = ([tuple(k) for k in keys], legs, int(rd_step))
        self._split = None
        if parallel_split_indices is not None:
            # reference: one MPI rank per tuple of consecutive sites (simulator_cls.py:243-249, _const_cls.py:236-251);
            # here one torch.distributed rank (= one GPU) per tuple, launched by torchrun
            if restart or self.model.one_gate_to_apply is not None or self.model.kraus_op is not None:  # noqa: SIM102
                raise NotImplementedError("site-parallel propagation supports neither restart nor gates / Kraus maps")
            self._split = [tuple(int(i) for i in seg) for seg in parallel_split_indices]
        return self._run(Δt if Δt is not None else stepsize, maxstep, False, restart, savefile_ext, loadfile_ext,
                         backup_interval, autocorr=autocorr, energy=energy, norm=norm, populations=populations,
                         observables=observables, thresh_sil=thresh_sil, integrator=integrator,
                         display_time_unit=display_time_unit, conserve_norm=conserve_norm, write_files=write_files,
                         record_trace=record_trace, suffix="_prop", adaptive=adaptive, p_svd=adaptive_p_svd,
                         adaptive_params=(adaptive_Dmax, adaptive_dD, adaptive_p_proj),
                         per_step=(autocorr_per_step, energy_per_step, norm_per_step, populations_per_step, observables_per_step))

    def _run(self, stepsize_fs, maxstep, relax, restart, savefile_ext, loadfile_ext, backup_interval, *, autocorr, energy,
             norm, populations, observables, thresh_sil, integrator, display_time_unit, conserve_norm, write_files,
             record_trace, suffix, adaptive=False, p_svd=1.0e-07, adaptive_params=(20, 5, 1.0e-04), per_step=(1, 1, 1, 1, 1)):
        autocorr_per_step, energy_per_step, norm_per_step, populations_per_step, observables_per_step = per_step
        stepsize_au = stepsize_fs / units.au_in_fs
        cfg = RunConfig(jobname=self.jobname + suffix, relax=relax, maxstep=maxstep, thresh_exp=thresh_sil,
                        verbose=self.verbose, space=self.model.space, integrator=integrator, conserve_norm=conserve_norm,
                        display_time_unit=display_time_unit, adaptive=adaptive, p_svd=p_svd, Dmax=int(adaptive_params[0]),
                        dD=int(adaptive_params[1]), p_proj=float(adaptive_params[2]))
        if not relax and getattr(self, "_two_site", (False, 0.0))[0]:
            cfg.two_site, cfg.two_site_p_svd = True, self._two_site[1]
            cfg.bond_dim = int(self.model.m_aux_max or 0)
        self._two_site = (False, 0.0)
        self.cfg = cfg
        split = getattr(self, "_split", None) if not relax else None
        if split is not None:
            wf = self._distributed_wavefunction(split)
            write_files = write_files and wf.ci_coef.rank == 0
            savefile_ext += f"_rank{wf.ci_coef.rank}"
        else:
            wf = self.get_initial_wavefunction(restart, loadfile_ext)
        wf.ci_coef.record_trace = record_trace
        # opt-in for the launch-bound regime (D <= 64, several whole-chain MPO keys): ``sim.merge_mpo_terms = True`` makes
        # DeviceMPO build one direct-sum MPO, i.e. one GEMM chain per apply instead of one per key.  Off by default because
        # the order of the term sum then differs from the reference's (results agree to ~1e-11 instead of ~1e-14); not
        # available for adaptive / site-parallel runs, whose bookkeeping addresses the keys individually.
        wf.merge_mpo_terms = bool(getattr(self, "merge_mpo_terms", False)) and split is None and not adaptive
        self.history = []
        files = self._open_files(cfg) if write_files else None
        if write_files:
            self.save_wavefunction(wf, savefile_ext)
        ham = self.model.hamiltonian
        time_au = cfg.time_au_init
        last_energy = None
        elapsed = 0.0
        for istep in range(maxstep):
            if write_files and istep % backup_interval == backup_interval - 1:
                self.save_wavefunction(wf, savefile_ext)
            rec: dict = {"time_au": time_au}
            if autocorr and istep % autocorr_per_step == 0:
                rec["autocorr"] = wf.autocorr()
            if energy and istep % energy_per_step == 0:
                rec["energy"] = last_energy = wf.expectation(ham)
            if norm and istep % norm_per_step == 0:
                rec["norm"] = wf.norm()
            if populations and istep % populations_per_step == 0:
                rec["pops"] = wf.pop_states()
            if observables and istep % observables_per_step == 0:
                rec["expectations"] = {k: wf.expectation(op) for k, op in self.model.observables.items()}
            if cfg.adaptive or cfg.two_site:
                rec["bonddim"] = wf.bonddim()
            rd = getattr(self, "_rd", None)
            if rd is not None and not relax and istep % rd[2] == 0:
                dens = wf.get_reduced_densities(rd[1])        # site-parallel runs: a collective call, values on rank 0
                if dens is not None:
                    rec["reduced_densities"] = dict(zip(rd[0], dens, strict=True))
            self.history.append(rec)
            if files is not None:
                self._export(files, cfg, rec, elapsed)
            t0 = _time.perf_counter()
            wf.propagate_SM(ham, stepsize_au, cfg, one_gate_to_apply=None if relax else self.model.one_gate_to_apply,
                            kraus_op=None if relax else self.model.kraus_op)
            elapsed += _time.perf_counter() - t0
            time_au += stepsize_au
        if files is not None:
            self.save_wavefunction(wf, savefile_ext)
            for f in files.values():
                f.close()
            rows = [r for r in self.history if "reduced_densities" in r]
            if rows:   # the reference writes <job>/reduced_density.nc (netCDF4); same content as an .npz here
                out = {"time_au": np.array([r["time_au"] for r in rows])}
                for key in rows[0]["reduced_densities"]:
                    out["rho_" + "_".join(map(str, key))] = np.stack([r["reduced_densities"][key] for r in rows])
                np.savez(os.path.join(cfg.jobname, "reduced_density.npz"), **out)
                _write_reduced_density_nc(os.path.join(cfg.jobname, "reduced_density.nc"), rows, display_time_unit)
        return (last_energy, wf)

    def relax(self, stepsize: float = 0.1, maxstep: int = 20, improved: bool = True, restart: bool = False,
              savefile_ext: str = "_gs", loadfile_ext: str = "", backup_interval: int = 10, norm: bool = True,
              populations: bool = True, observables: bool = False, integrator: str = "lanczos",
              display_time_unit: str = "fs", write_files: bool = True, record_trace: bool = False,
              two_site: bool = False):
        """Ground-state relaxation (reference ``simulator_cls.py:95-158``): improved relaxation (per-site Lanczos
        eigen-solve, default) or imaginary-time propagation.  Returns ``(energy, wf)``.  One-site only."""
        if two_site:
            raise NotImplementedError("two-site relaxation is not implemented; relax runs the one-site scheme")
        return self._run(stepsize, maxstep, "improved" if improved else True, restart, savefile_ext, loadfile_ext,
                         backup_interval, autocorr=False, energy=True, norm=norm, populations=populations,
                         observables=observables, thresh_sil=1.0e-09, integrator=integrator,
                         display_time_unit=display_time_unit, conserve_norm=True, write_files=write_files,
                         record_trace=record_trace, suffix="_relax")

    def operate(self, maxstep: int = 10, restart: bool = False, savefile_ext: str = "_operate", loadfile_ext: str = "_gs",
                verbose: int = 2, write_files: bool = True, two_site: bool = False):
        """Apply the model's ``hamiltonian`` entry -- in this mode an operator such as a dipole MPO -- to the wavefunction
        (reference ``Simulator.operate``, simulator_cls.py:286-330, 356-361): |Psi'> = O|Psi> / |O|Psi>|.  Returns
        ``(|O|Psi>|, wf)`` and writes ``wf_<jobname><savefile_ext>.pkl``, from which ``propagate(restart=True, loadfile_ext=
        savefile_ext)`` continues -- the relax -> operate -> propagate workflow of the reference's spectra notebooks."""
        if two_site:
            raise NotImplementedError("operate fits O|Psi> with one-site sweeps; there is no two-site variant")
        if self.model.space != "hilbert":
            raise NotImplementedError("operate is implemented for Hilbert-space MPS")
        wf = self.get_initial_wavefunction(restart, loadfile_ext)
        jobdir = self.jobname + "_operate"
        log = None
        f = None
        if write_files:
            os.makedirs(jobdir, exist_ok=True)
            f = _DatFile(os.path.join(jobdir, "main.log"))
            f.write("Start: apply operator to wave function")
            if verbose > 1:
                log = f.write
        norm = wf.apply_dipole(self.model.hamiltonian, maxstep=maxstep, log=log)
        if write_files:
            self.save_wavefunction(wf, savefile_ext)
            f.write(f"End  : apply operator to wave function, norm = {norm}")
            f.close()
        return (norm, wf)

    # -- output files in the reference's layout (properties.py:287-356) -----------------------------
    def _open_files(self, cfg: RunConfig) -> dict:
        os.makedirs(cfg.jobname, exist_ok=True)
        return {name: _DatFile(os.path.join(cfg.jobname, fn)) for name, fn in
                (("main", "main.log"), ("auto", "autocorr.dat"), ("pop", "populations.dat"), ("exp", "expectations.dat"))
                + ((("bond", "bonddim.dat"),) if cfg.adaptive or cfg.two_site else ())}

    def _export(self, files: dict, cfg: RunConfig, rec: dict, elapsed: float):
        unit = cfg.display_time_unit
        t = rec["time_au"] * {"au": 1.0, "fs": units.au_in_fs, "ps": units.au_in_fs * 1e-3}[unit]
        first = rec["time_au"] == cfg.time_au_init
        if "autocorr" in rec:
            if first:
                files["auto"].write(f"# time [{unit}]\t auto-correlation")
            a = rec["autocorr"]
            files["auto"].write(f"{2 * t:6.9f}\t{a.real: 6.9f}{a.imag:+6.9f}j")
        if "pops" in rec:
            if first:
                files["pop"].write(f"# time [{unit}]\t" + "\t".join(f"pop_{i}".ljust(11) for i in range(len(rec["pops"]))))
            files["pop"].write(f"{t:6.9f}\t" + "".join(f"{p:6.9f}\t" for p in rec["pops"]))
        if "bonddim" in rec and "bond" in files:     # adaptive and two-site runs: properties.py:344-356
            if first:
                files["bond"].write(f"# time [{unit}]\t" + "\t".join(f"{i}" for i in range(len(rec["bonddim"]))))
            files["bond"].write(f"{t:6.9f}\t" + "".join(f"{b}\t" for b in rec["bonddim"]))
        if rec.get("expectations"):
            if first:
                files["exp"].write(f"# time [{unit}]\t" + "\t".join(str(k).ljust(11) for k in rec["expectations"]))
            files["exp"].write(f"{t:6.9f}\t" + "".join(f"{v:6.9f}\t" for v in rec["expectations"].values()))
        if cfg.verbose > 1:
            msg = ""
            if "autocorr" in rec:
                msg += f"| autocorr: {rec['autocorr'].real: 6.4f}{rec['autocorr'].imag:+6.4f}i"
            if "pops" in rec:
                msg += "| pop" + "".join(f" {p:6.4f} " for p in rec["pops"][:3])
            if "energy" in rec:
                msg += f"| ene[eV]: {np.real(rec['energy']) * units.au_in_eV:10.7f} "
            msg += f"| time[{unit}]: {t:8.3f} | elapsed[sec]:{elapsed:9.2f} "
            files["main"].write(msg)
