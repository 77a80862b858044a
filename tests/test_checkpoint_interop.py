"""Checkpoint / MPO interoperability with the reference's file formats (SURVEY 8(f4); pytdscf/simulator_cls.py:501-507,
:577-589; pympo.utils.import_npz).  Fixture made by tests/golden/make_golden_checkpoint.py with the unmodified reference:
its exciton state after 3 steps and the energies of the reference continuing from it."""
import os
import pickletools

import numpy as np
import pytest

from tests.golden_io import load_checkpoint, load_run, write_checkpoint


def test_read_reference_pickle_without_the_reference_installed(tmp_path):
    """The reference's state after 3 steps in its ``wf_*.pkl`` format (``tests.golden_io.write_checkpoint``; the reference
    continued from such a file exactly as from its own dump) reads back without the reference installed."""
    import sys

    from pytdscf_b200.checkpoint import is_reference_pickle, read_reference_wavefunction

    path = write_checkpoint(str(tmp_path / "wf_ck.pkl"))
    names = {arg for op, arg, _ in pickletools.genops(open(path, "rb").read()) if op.name == "SHORT_BINUNICODE" and isinstance(arg, str)}
    for module, cls in [("pytdscf.wavefunction", "WFunc"), ("pytdscf._mps_mpo", "MPSCoefMPO"), ("pytdscf._mps_cls", "LatticeInfo"),
                        ("pytdscf._site_cls", "SiteCoef"), ("pytdscf._spf_cls", "SPFCoef")]:
        assert module in names and cls in names
    assert "pytdscf" not in sys.modules or not hasattr(sys.modules["pytdscf"], "Simulator")  # really not the reference
    assert is_reference_pickle(path)
    d = read_reference_wavefunction(path)
    z = load_checkpoint()
    assert d["gauges"] == [str(g) for g in z["gauges"]] == ["Psi", "B", "B", "B"]
    for i, c in enumerate(d["cores"]):
        assert c.dtype == np.complex128 and (c == z[f"core{i}"]).all()
    # tests/golden/make_golden_checkpoint.py: the reference restarted from such a file reproduces its own continuation
    assert (z["energies_restart_our_file"] == z["energies_restart_reference_file"]).all()


def test_restart_from_a_reference_checkpoint_host_logic(tmp_path):
    """Simulator(restart=True) picks up a wf_*.pkl in the reference's format (``tests.golden_io.write_checkpoint``) and
    continues like the reference does (CPU host logic with the oracle's kernels; the GPU version is in
    tests/test_gpu_propagation.py)."""
    import pytdscf_b200 as tb
    from oracle.oracle_engine import OracleEngine
    from tests.test_host_sweep_cpu import _build_model

    g = load_run("exciton_D6")
    os.chdir(tmp_path)
    write_checkpoint("wf_ck.pkl")
    sim = tb.Simulator("ck", _build_model(g), backend="cuda", verbose=0)
    sim.eng = OracleEngine()
    ener, wf = sim.propagate(stepsize=0.1, maxstep=3, restart=True, loadfile_ext="", savefile_ext="_cont", autocorr=False,
                             norm=False, populations=False)
    ref = load_checkpoint()["energies_restart_reference_file"]
    got = [rec["energy"] for rec in sim.history]
    assert np.allclose(got, ref, rtol=0, atol=1e-13)
    # and hand the result back in the reference's format
    out = sim.save_wavefunction(wf, "_ref", reference_format=True)
    from pytdscf_b200.checkpoint import is_reference_pickle

    assert is_reference_pickle(out)


def test_mpo_npz_import_export(tmp_path):
    import pytdscf_b200 as tb

    g = load_run("exciton_D2")
    (key, cores), = [(k, v) for k, v in g["operators"].items() if len(k) == 4]
    path = tb.export_mpo_npz(str(tmp_path / "mpo.npz"), cores)
    assert sorted(np.load(path).files) == ["W0", "W1", "W2", "W3"]             # the pympo.utils.export_npz layout
    back = tb.import_mpo_npz(path)
    assert len(back) == 4 and all((a == b).all() for a, b in zip(back, cores, strict=True))
    tb.TensorOperator(mpo=back)                                                 # usable as MPO cores right away
    np.savez(str(tmp_path / "pos.npz"), *cores)                                 # np.savez positional layout
    assert all((a == b).all() for a, b in zip(tb.import_mpo_npz(str(tmp_path / "pos.npz")), cores, strict=True))
    np.savez(str(tmp_path / "bad.npz"), W0=cores[0], W2=cores[1])
    with pytest.raises(ValueError):
        tb.import_mpo_npz(str(tmp_path / "bad.npz"))
    np.savez(str(tmp_path / "bond.npz"), W0=cores[0], W1=cores[2])
    with pytest.raises(ValueError):
        tb.import_mpo_npz(str(tmp_path / "bond.npz"))
