"""bench.py's contract: on the CPU the reference arm's JSON line and the refusal of the product arm to run (or fall back) without
a device; on the GPU the number of timed steps and the outputs --dump-outputs writes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--genes", "400", "--samples", "24", "--cpu-sample-genes", "200")
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "genes/s" and line["higher_is_better"] is True
    assert line["metric"].startswith("genes/sec") and line["value"] > 0 and line["steps"] == 1 and line["n_gpus"] == 1
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "genes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and line["scaling"] == "weak" and line["dtype"] == "f64"


def test_product_arm_fails_loudly_without_a_gpu():
    import ctypes

    try:  # a visible CUDA device means this is the GPU box: nothing to check here
        if ctypes.CDLL("libcuda.so.1").cuInit(0) == 0:
            n = ctypes.c_int(0)
            ctypes.CDLL("libcuda.so.1").cuDeviceGetCount(ctypes.byref(n))
            if n.value > 0:
                return
    except OSError:
        pass
    r = _run("--steps", "1", "--warmup", "1", "--genes", "200", "--samples", "12", "--no-cpu-baseline")
    assert r.returncode != 0
    assert "no CPU fallback" in r.stderr and not r.stdout.strip().startswith("{")


def test_steps_below_one_are_refused():
    r = _run("--impl", "reference", "--steps", "0")
    assert r.returncode != 0 and "--steps must be at least 1" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step_and_repeat(tmp_path):
    """--steps sets the timed steps; --dump-outputs writes the headline pass' tables as float64 .npy, the same on a second run and
    the same as one pass of the library over the same seeded workload."""
    args = ["--steps", "2", "--warmup", "1", "--genes", "3000", "--samples", "24", "--no-cpu-baseline", "--no-extra-configs"]
    dumps = []
    for i in range(2):
        d = tmp_path / f"run{i}"
        r = _run(*args, "--dump-outputs", str(d))
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2 and len(line["e2e"]["step_wall_ms"]) == len(line["e2e"]["pageable"]["step_wall_ms"]) == 2
        dumps.append({f.stem: np.load(f) for f in sorted(d.glob("*.npy"))})
    a, b = dumps
    assert {"lfc", "se", "stat", "pvalue", "dispersions", "genewise", "map", "trend_coeffs"} <= set(a) and set(a) == set(b)
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    G = a["dispersions"].shape[0]
    assert 2000 < G <= 3000 and a["lfc"].shape == (G, 2)
    for k in a:
        assert a[k].dtype == np.float64
        np.testing.assert_allclose(a[k], b[k], rtol=1e-12, atol=0, equal_nan=True, err_msg=k)
    from bench import make_workload
    from pydeseq2_b200.inference import B200Inference
    from pydeseq2_b200.pipeline import ResidentFit

    counts, X, sf, _ = make_workload(24, 3000, "two_level", 0)
    rf = ResidentFit(B200Inference(device=0)._ops.ctx, X, sf)
    rf.upload(counts)
    want = rf.run()
    rf.close()
    for k in ("dispersions", "genewise", "lfc", "se", "pvalue"):
        np.testing.assert_allclose(a[k], want[k], rtol=1e-9, atol=0, equal_nan=True, err_msg=k)


def test_dump_outputs_samples_genes_above_the_bound(tmp_path):
    import types

    from bench import dump_outputs

    G, rng = 5000, np.random.default_rng(1)
    res = {"dispersions": rng.random(G), "lfc": rng.random((G, 2)), "pvalue": rng.random(G), "prior_var": 0.3,
           "squared_logres": 1.2, "trend": types.SimpleNamespace(coeffs=np.array([0.1, 2.0]))}
    dump_outputs(tmp_path / "full", res)
    full = {f.stem: np.load(f) for f in (tmp_path / "full").glob("*.npy")}
    assert "gene_index" not in full and full["lfc"].shape == (G, 2) and full["prior_var"].tolist() == [0.3]
    limit = 1 << 17  # 32 bytes per gene: 160 000 bytes in all
    for run in ("a", "b"):
        dump_outputs(tmp_path / run, res, limit=limit)
    files = sorted((tmp_path / "a").glob("*.npy"))
    assert sum(f.stat().st_size for f in files) <= limit
    got = {f.stem: np.load(f) for f in files}
    idx = got["gene_index"].astype(np.int64)
    assert 1000 < len(idx) < G and (np.diff(idx) > 0).all()
    np.testing.assert_array_equal(got["lfc"], res["lfc"][idx])
    np.testing.assert_array_equal(got["pvalue"], res["pvalue"][idx])
    np.testing.assert_array_equal(got["trend_coeffs"], [0.1, 2.0])
    np.testing.assert_array_equal(idx, np.load(tmp_path / "b" / "gene_index.npy"))  # the sample is fixed
