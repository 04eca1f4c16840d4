"""Helper of tests/test_reference_dropin.py, run in a SUBPROCESS: the REAL, unmodified orchestrator of the
reference (`DeseqDataSet.deseq2()`, `DeseqStats.summary()`, `lfc_shrink()`) with `B200Inference` injected as its `inference=`
backend -- device algorithms through the host emulator, so no GPU is needed.  Writes the final tables to an .npz.
The import shims (oracle/refshim*) stay inside this process."""
import os
import sys
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for d in ("refshim", "refshim_orch"):
    sys.path.insert(0, os.path.join(ROOT, "oracle", d))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import pandas as pd  # noqa: E402


def main(fixture, out, subclass=False):
    from pydeseq2.dds import DeseqDataSet
    from pydeseq2.ds import DeseqStats
    from pydeseq2.inference import Inference

    from emu.emu_ops import EmuOps
    from pydeseq2_b200.inference import B200Inference

    assert issubclass(B200Inference, Inference)       # with the reference importable the backend IS a pydeseq2 Inference
    g = np.load(fixture)
    counts, X, contrast = g["counts"], g["design"], g["contrast"]
    N, G = counts.shape
    idx = [f"s{i}" for i in range(N)]
    counts_df = pd.DataFrame(counts, index=idx, columns=[f"g{i}" for i in range(G)])
    design_df = pd.DataFrame(X, index=idx, columns=[f"x{j}" for j in range(X.shape[1])])
    meta = pd.DataFrame({"dummy": np.arange(N)}, index=idx)
    backend = B200Inference(_ops=EmuOps())
    if subclass:   # size factors and Cook's distances through the backend as well (pydeseq2_b200/integration.py)
        from pydeseq2_b200.integration import b200_dataset_class

        DeseqDataSet = b200_dataset_class()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        dds = DeseqDataSet(counts=counts_df, metadata=meta, design=design_df, inference=backend, quiet=True)
        dds.deseq2()
        ds = DeseqStats(dds, contrast=contrast, inference=backend, quiet=True)
        ds.summary()
        res = ds.results_df.copy()   # lfc_shrink() below overwrites columns of results_df in place
        k = int(np.flatnonzero(contrast)[-1])
        # ds.lfc_shrink() itself: under pandas 3 its `.iloc[:, k].update(...)` writes into a temporary (oracle/make_golden.py notes
        # the same for the reference's own backend), so the plugin call is what is checked here
        size = 1.0 / dds.var["dispersions"].values
        offset = np.log(dds.obs["size_factors"]).values
        nz = dds.non_zero_idx
        prior_var = ds._fit_prior_var(coeff_idx=k)
        ds.lfc_shrink(coeff=design_df.columns[k])
        shrunk = backend.lfc_shrink_nbinom_glm(design_matrix=X, counts=dds.X[:, nz], size=size[nz], offset=offset,
                                              prior_no_shrink_scale=15, prior_scale=float(np.minimum(np.sqrt(prior_var), 1)),
                                              optimizer="L-BFGS-B", shrink_index=k)
    # the variance-stabilising transformation, another caller of the same plugin methods (dds.py:349-515: intercept-only design,
    # `fit_genewise_dispersions(vst=True)` + trend fit, then a closed-form transform): through the backend under test and through
    # the reference's own CPU backend, in this process
    from oracle.make_golden import ref_inference

    vst = {}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for tag, inf in (("b200", backend), ("ref", ref_inference())):
            cls = DeseqDataSet if tag == "b200" else __import__("pydeseq2.dds", fromlist=["DeseqDataSet"]).DeseqDataSet
            for fit_type in ("parametric", "mean"):
                d2 = cls(counts=counts_df, metadata=meta, design=design_df, inference=inf, quiet=True)
                d2.vst(fit_type=fit_type)
                vst[f"vst_{fit_type}_{tag}"] = np.asarray(d2.layers["vst_counts"], dtype=float)
            # transform of held-out counts with the FITTED log means (the override must have stored them: dds.py:438-480)
            vst[f"vst_new_{tag}"] = np.asarray(d2.vst_transform(counts[: N // 2] + 1), dtype=float)
    np.savez(out, **vst, baseMean=res["baseMean"].values, log2FoldChange=res["log2FoldChange"].values, lfcSE=res["lfcSE"].values,
             stat=res["stat"].values, pvalue=res["pvalue"].values, padj=res["padj"].values, LFC=dds.varm["LFC"].values,
             dispersions=dds.var["dispersions"].values, replaced=np.asarray(dds.var["replaced"], dtype=float),
             cooks_outlier=np.asarray(dds.cooks_outlier(), dtype=float), shrunk_lfc=shrunk[0], shrink_converged=shrunk[2],
             shrink_flag_set=np.float64(ds.shrunk_LFCs), n_cpus=np.float64(backend.n_cpus or 0))


def variants(fixture, out):
    """Two more ways the reference's orchestrator drives the same plugin calls, each through the backend under test and through
    the reference's own CPU backend: (a) the iterative size-factor estimator it switches to when every gene holds a zero
    (dds.py:682-690, 1460-1545: rounds of genewise / MAP dispersion fits on an intercept-only design around a Powell search) --
    reached here through the subclass, whose device median-of-ratios raises the same ValueError first; (b) `low_memory=True`
    (dds.py:934, 1032, 1103: (N, G) intermediates are dropped as soon as they are used)."""
    from pydeseq2.dds import DeseqDataSet
    from pydeseq2.ds import DeseqStats

    from emu.emu_ops import EmuOps
    from oracle.make_golden import ref_inference
    from pydeseq2_b200.inference import B200Inference
    from pydeseq2_b200.integration import b200_dataset_class

    g = np.load(fixture)
    counts, X, contrast = g["counts"][:, :120], g["design"], g["contrast"]
    N, G = counts.shape
    idx = [f"s{i}" for i in range(N)]
    design_df = pd.DataFrame(X, index=idx, columns=[f"x{j}" for j in range(X.shape[1])])
    meta = pd.DataFrame({"dummy": np.arange(N)}, index=idx)
    with_zero = counts.copy()
    with_zero[np.random.default_rng(3).integers(0, N, G), np.arange(G)] = 0  # a zero in every gene
    res = {}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for tag, cls, inf in (("b200", b200_dataset_class(), B200Inference(_ops=EmuOps())), ("ref", DeseqDataSet, ref_inference())):
            df = pd.DataFrame(with_zero, index=idx, columns=[f"g{i}" for i in range(G)])
            d = cls(counts=df, metadata=meta, design=design_df, inference=inf, quiet=True)
            d.fit_size_factors()
            res["iterative_sf_" + tag] = np.asarray(d.obs["size_factors"], dtype=float)
            df = pd.DataFrame(counts, index=idx, columns=[f"g{i}" for i in range(G)])
            d = cls(counts=df, metadata=meta, design=design_df, inference=inf, quiet=True, low_memory=True)
            d.deseq2()
            st = DeseqStats(d, contrast=contrast, inference=inf, quiet=True)
            st.summary()
            for col in ("log2FoldChange", "lfcSE", "pvalue", "padj"):
                res[f"lowmem_{col}_{tag}"] = st.results_df[col].values.astype(float)
            res["lowmem_kept_" + tag] = np.float64(sum(k.startswith("_") for k in list(d.layers.keys()) + list(d.obsm.keys())))
    np.savez(out, **res)


if __name__ == "__main__":
    if len(sys.argv) > 3 and sys.argv[3] == "variants":
        variants(sys.argv[1], sys.argv[2])
    else:
        main(sys.argv[1], sys.argv[2], subclass=len(sys.argv) > 3 and sys.argv[3] == "subclass")
