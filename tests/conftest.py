import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")
    config.addinivalue_line("markers", "refcheck: needs the reference package build() byte-compiles into oracle/_ref")


def load_golden(name):
    with np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False) as z:
        return {k: z[k] for k in z.files}


@pytest.fixture(scope="session")
def golden():
    return load_golden


def tape_calls(t):
    """Decode a tape_*.npz into [(method, kwargs, outs)] in call order."""
    calls = []
    for i in range(int(t["n_calls"])):
        keys = sorted(k for k in t if k.startswith(f"c{i:02d}_"))
        meth = keys[0].split("__")[0][4:]
        kw, args, outs = {}, {}, {}
        for k in keys:
            field = k.split("__")[1]
            v = t[k]
            if field.startswith("out"):
                outs[int(field[3:])] = v
            elif field.startswith("arg"):
                args[int(field[3:])] = v
            elif field == "alt_hypothesis":
                kw[field] = str(v) or None
            elif field in ("cr_reg", "prior_reg"):
                kw[field] = bool(v)
            elif field in ("min_mu", "beta_tol", "min_disp", "max_disp", "prior_disp_var", "lfc_null"):
                kw[field] = None if np.isnan(v).all() else float(np.ravel(v)[0])
            else:
                kw[field] = v
        if "counts" in kw:
            kw["counts"] = kw["counts"].astype(np.int64)
        calls.append((meth, [args[j] for j in sorted(args)], kw, [outs[j] for j in sorted(outs)]))
    return calls
