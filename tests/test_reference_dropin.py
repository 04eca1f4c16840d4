"""CPU suite: `B200Inference` plugged into the REAL reference orchestrator (`DeseqDataSet(..., inference=)`,
`DeseqStats(..., inference=)`), i.e. the drop-in claim of INTEGRATION.md exercised with the reference's own objects.  The device
algorithms run through the host emulator.  The reference package is the byte-compiled copy build() leaves in oracle/_ref."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, load_golden

HERE = os.path.dirname(os.path.abspath(__file__))
REF_PKG = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "pydeseq2")
pytestmark = [pytest.mark.refcheck,
              pytest.mark.skipif(not os.path.isfile(os.path.join(REF_PKG, "dds.pyc")),
                                 reason="the reference package was not compiled into oracle/_ref (build() found no reference checkout)")]


@pytest.mark.parametrize("name,mode", [("e2e_two_level_n24", "plugin"), ("e2e_factorial_n20", "plugin"),
                                       ("e2e_two_level_n24", "subclass"), ("e2e_factorial_n20", "subclass")])
def test_real_orchestrator_with_b200_backend(name, mode, tmp_path):
    """mode "plugin": the stock DeseqDataSet with `inference=B200Inference`; mode "subclass": `integration.b200_dataset_class()`,
    which also routes size factors and Cook's distances through the backend."""
    out = str(tmp_path / "res.npz")
    env = dict(os.environ)
    env.pop("PYTHONPATH", None)
    r = subprocess.run([sys.executable, os.path.join(HERE, "dropin_reference_run.py"), os.path.join(GOLDEN, name + ".npz"), out, mode],
                       capture_output=True, text=True, timeout=1500, env=env)
    assert r.returncode == 0, r.stderr[-3000:]
    got, ref = np.load(out), load_golden(name)
    # discrete outcomes of the orchestrator equal those it reached with its own CPU backend
    np.testing.assert_array_equal(got["replaced"], ref["final_replaced"])
    np.testing.assert_array_equal(got["cooks_outlier"], ref["final_cooks_outlier"])
    np.testing.assert_array_equal(np.isnan(got["pvalue"]), np.isnan(ref["final_pvalue"]))
    np.testing.assert_array_equal(np.isnan(got["padj"]), np.isnan(ref["final_padj"]))
    np.testing.assert_allclose(got["baseMean"], ref["final_baseMean"], rtol=1e-12)

    def mostly(a, b, rtol, atol=0.0):  # same mismatch budget as tests/parity.py::check_e2e
        bad = ~np.isclose(a, b, rtol=rtol, atol=atol, equal_nan=True)
        assert bad.mean() <= 0.005, bad.mean()
        np.testing.assert_allclose(a, b, rtol=100 * rtol, atol=100 * atol, equal_nan=True)

    mostly(got["LFC"], ref["final_LFC"], 1e-4, 1e-8)
    mostly(got["dispersions"], ref["final_dispersions"], 1e-4)
    mostly(got["log2FoldChange"], ref["final_log2FoldChange"], 1e-4, 1e-8)
    mostly(got["lfcSE"], ref["final_lfcSE"], 1e-4)
    mostly(got["stat"], ref["final_stat"], 1e-4, 1e-8)
    big = ref["final_pvalue"] >= 1e-20
    mostly(got["pvalue"][big], ref["final_pvalue"][big], 1e-3)
    ok = ~np.isnan(ref["final_padj"]) & big
    mostly(got["padj"][ok], ref["final_padj"][ok], 1e-3)
    # vst(): same transformed counts as with the reference's CPU backend (the trend coefficients come from two different
    # minimisers of the same objective, ~4e-6 apart: SURVEY App. B)
    for key in ("vst_parametric", "vst_mean", "vst_new"):
        np.testing.assert_allclose(got[key + "_b200"], got[key + "_ref"], rtol=2e-5, atol=1e-6)
    # the shrinkage plugin call made by the orchestrator's own lfc_shrink() went through the backend
    assert got["shrink_flag_set"] == 1.0 and got["shrink_converged"].mean() > 0.99
    assert np.isfinite(got["shrunk_lfc"]).all()
    assert got["n_cpus"] > 0   # the orchestrator set the attribute it expects on a backend (dds.py:323-333)


def test_real_orchestrator_variants_with_b200_backend(tmp_path):
    """Iterative size factors (every gene holds a zero) and `low_memory=True`: the orchestrator's other routes through the same
    plugin calls give the reference CPU backend's numbers with the B200 backend."""
    out = str(tmp_path / "variants.npz")
    env = dict(os.environ)
    env.pop("PYTHONPATH", None)
    r = subprocess.run([sys.executable, os.path.join(HERE, "dropin_reference_run.py"), os.path.join(GOLDEN, "e2e_two_level_n24.npz"), out,
                        "variants"], capture_output=True, text=True, timeout=1500, env=env)
    assert r.returncode == 0, r.stderr[-3000:]
    got = np.load(out)
    np.testing.assert_allclose(got["iterative_sf_b200"], got["iterative_sf_ref"], rtol=1e-5)
    assert got["lowmem_kept_b200"] == got["lowmem_kept_ref"] == 0  # the (N, G) intermediates were dropped on both sides
    np.testing.assert_array_equal(np.isnan(got["lowmem_padj_b200"]), np.isnan(got["lowmem_padj_ref"]))
    np.testing.assert_allclose(got["lowmem_log2FoldChange_b200"], got["lowmem_log2FoldChange_ref"], rtol=1e-4, atol=1e-8)
    np.testing.assert_allclose(got["lowmem_lfcSE_b200"], got["lowmem_lfcSE_ref"], rtol=1e-4)
    np.testing.assert_allclose(got["lowmem_pvalue_b200"], got["lowmem_pvalue_ref"], rtol=1e-3)
    np.testing.assert_allclose(got["lowmem_padj_b200"], got["lowmem_padj_ref"], rtol=1e-3)
