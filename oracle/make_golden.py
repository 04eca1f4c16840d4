"""Generate the golden vectors under tests/golden/ from the REAL reference.  TEST INFRASTRUCTURE.

Runs only in the build container (needs the read-only checkout at /root/reference, imported
through ``oracle/refshim`` + ``oracle/refshim_orch``; see SURVEY.md Appendix A).  The outputs
are small ``.npz`` files that travel to the GPU box, where the reference does not exist.

    python oracle/make_golden.py            # rewrites tests/golden/*.npz

Two kinds of fixture:

* ``calls_*.npz``  -- seeded synthetic inputs pushed through every hot-path method of the
  reference's ``DefaultInference`` (per-call isolation parity);
* ``tape_*.npz``   -- every ``Inference`` call (inputs AND outputs) the reference's own
  ``DeseqDataSet.deseq2()`` + ``DeseqStats.summary()`` make on the datasets shipped with the
  reference, plus the final LFC/dispersion/p-value tables and the stored R DESeq2 results
  (``tests/data/**/r_test_res.csv``) for those datasets.
"""
from __future__ import annotations

import os
import sys
import warnings

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for d in ("refshim", "refshim_orch"):
    sys.path.insert(0, os.path.join(HERE, d))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import pandas as pd  # noqa: E402

REF = "/root/reference"
OUT = os.path.join(ROOT, "tests", "golden")


def synth(N, G, design, seed=0, mean_log2=4.0):
    """SURVEY.md §8(d) generator (DESeq2 makeExampleDESeqDataSet-like)."""
    from pydeseq2_b200.synth import make_counts

    return make_counts(N, G, design, seed, mean_log2=mean_log2)


def ref_inference():
    from pydeseq2.default_inference import DefaultInference

    class FloatFlags(DefaultInference):
        """pandas-3 compatibility: converged as float (SURVEY.md §8c)."""

        def irls(self, *a, **k):
            b, m, h, c = super().irls(*a, **k)
            return b, m, h, np.asarray(c, dtype=float)

        def alpha_mle(self, *a, **k):
            d, c = super().alpha_mle(*a, **k)
            return d, np.asarray(c, dtype=float)

    return FloatFlags(n_cpus=1)


def gen_calls(name, N, G, design_kind, seed, mean_log2=4.0):
    from pydeseq2.preprocessing import deseq2_norm

    inf = ref_inference()
    counts, X, _truth = synth(N, G, design_kind, seed, mean_log2)
    # drop all-zero genes like dds.py:729-731
    counts = counts[:, ~(counts == 0).all(0)]
    normed, sf = deseq2_norm(counts)
    p = X.shape[1]
    out = dict(counts=counts, X=X, sf=sf, normed=normed)
    out["rough"] = inf.fit_rough_dispersions(normed, pd.DataFrame(X))
    out["moments"] = inf.fit_moments_dispersions(normed, sf)
    max_disp = max(10.0, N)
    mom = np.clip(np.minimum(out["rough"], out["moments"]), 1e-8, max_disp)
    out["mom"] = mom
    out["lin_mu"] = inf.lin_reg_mu(counts, sf, X, 0.5)
    b, m, h, c = inf.irls(counts, sf, X, mom, 0.5, 1e-8)
    out.update(irls0_beta=b, irls0_mu=np.ascontiguousarray(m), irls0_hat=np.ascontiguousarray(h), irls0_conv=c)
    mu_hat = np.ascontiguousarray(out["lin_mu"] if design_kind in ("two_level", "intercept") else m)
    out["mu_hat"] = mu_hat
    a, c = inf.alpha_mle(counts, X, mu_hat, mom, 1e-8, max_disp)
    out.update(gw_alpha=a, gw_conv=c)
    gw = np.clip(a, 1e-8, max_disp)
    # a synthetic "trend" for the MAP stage (any positive vector is a valid alpha_hat)
    rng = np.random.default_rng(seed + 1)
    trend = gw * np.exp(rng.normal(0, 0.3, gw.shape))
    out["trend"] = trend
    out["prior_var"] = np.float64(0.6)
    a, c = inf.alpha_mle(counts, X, mu_hat, trend, 1e-8, max_disp, prior_disp_var=0.6, cr_reg=True, prior_reg=True)
    out.update(map_alpha=a, map_conv=c)
    disp = np.clip(a, 1e-8, max_disp)
    out["disp"] = disp
    b, m, h, c = inf.irls(counts, sf, X, disp, 0.5, 1e-8)
    out.update(lfc_beta=b, lfc_mu=np.ascontiguousarray(m), lfc_hat=np.ascontiguousarray(h), lfc_conv=c)
    contrast = np.zeros(p)
    contrast[min(1, p - 1)] = 1.0
    ridge = np.diag(np.repeat(1e-6, p))
    out.update(contrast=contrast, ridge=ridge)
    mu_w = np.ascontiguousarray(m)
    for alt, null in ((None, 0.0), ("greater", 0.3), ("less", 0.3), ("greaterAbs", 0.3), ("lessAbs", 0.3)):
        pv, st, se = inf.wald_test(X, disp, b, mu_w, ridge, contrast, null, alt)
        tag = alt or "two_sided"
        out[f"wald_{tag}_p"], out[f"wald_{tag}_stat"], out[f"wald_{tag}_se"] = pv, st, se
    coeffs, pred, ok = inf.dispersion_trend_gamma_glm(pd.Series(1.0 / normed.mean(0)), pd.Series(gw))
    out.update(trend_coeffs=coeffs, trend_pred=pred, trend_ok=np.float64(ok))
    np.savez_compressed(os.path.join(OUT, f"calls_{name}.npz"), **out)
    print(f"calls_{name}: N={N} G={counts.shape[1]} p={p}")


class Tape:
    """Wraps an Inference and records every hot-path call."""

    def __init__(self, inner):
        self._inner = inner
        self.calls = []

    n_cpus = property(lambda s: s._inner.n_cpus, lambda s, v: setattr(s._inner, "n_cpus", v))

    def __getattr__(self, name):
        fn = getattr(self._inner, name)
        if name not in ("lin_reg_mu", "irls", "alpha_mle", "wald_test", "fit_rough_dispersions",
                        "fit_moments_dispersions", "dispersion_trend_gamma_glm"):
            return fn

        def rec(*a, **k):
            # snapshot the inputs NOW: the orchestrator hands out views of its own columns (e.g. `.values` of
            # var["fitted_dispersions"]) and overwrites them in place later (outlier refit, dds.py:1440-1458)
            snap = lambda v: v.copy() if hasattr(v, "copy") else v  # noqa: E731
            a0, k0 = tuple(snap(v) for v in a), {kk: snap(v) for kk, v in k.items()}
            res = fn(*a, **k)
            r0 = tuple(snap(v) for v in res) if isinstance(res, tuple) else snap(res)
            self.calls.append((name, a0, k0, r0))
            return res

        return rec


def _arr(v):
    if isinstance(v, (pd.Series, pd.DataFrame)):
        v = v.values
    if v is None:
        return np.array(np.nan)
    return np.ascontiguousarray(np.asarray(v, dtype=float) if not isinstance(v, str) else np.array(v))


def gen_tape(name, counts_df, metadata, design_df, contrast, r_res_csv, r_disp_csv=None, **dds_kwargs):
    from pydeseq2.dds import DeseqDataSet
    from pydeseq2.ds import DeseqStats

    tape = Tape(ref_inference())
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        dds = DeseqDataSet(counts=counts_df, metadata=metadata, design=design_df, inference=tape, quiet=True,
                           **dds_kwargs)
        dds.deseq2()
        ds = DeseqStats(dds, contrast=np.asarray(contrast, dtype=float), inference=tape, quiet=True)
        ds.summary()
    out = {}
    for i, (meth, a, k, res) in enumerate(tape.calls):
        pre = f"c{i:02d}_{meth}"
        assert not a or meth in ("fit_rough_dispersions", "fit_moments_dispersions", "dispersion_trend_gamma_glm")
        for j, v in enumerate(a):
            out[f"{pre}__arg{j}"] = _arr(v)
        for kk, v in k.items():
            if kk == "alt_hypothesis":
                out[f"{pre}__{kk}"] = np.array("" if v is None else v)
            elif kk in ("cr_reg", "prior_reg"):
                out[f"{pre}__{kk}"] = np.array(float(v))
            else:
                out[f"{pre}__{kk}"] = _arr(v)
        res = res if isinstance(res, tuple) else (res,)
        for j, v in enumerate(res):
            out[f"{pre}__out{j}"] = _arr(v)
    out["n_calls"] = np.array(len(tape.calls))
    out["final_LFC"] = dds.varm["LFC"].values
    out["final_dispersions"] = dds.var["dispersions"].values
    out["final_genewise"] = dds.var["genewise_dispersions"].values
    out["final_size_factors"] = dds.obs["size_factors"].values
    out["final_pvalues"] = ds.p_values.values
    out["final_stat"] = ds.statistics.values
    out["final_se"] = ds.SE.values
    out["final_padj"] = ds.padj.values
    # Cook's distances (dds.py:986-1040) and what the orchestrator derives from them
    from pydeseq2.utils import robust_method_of_moments_disp

    nzm = dds.var["non_zero"].values
    out["final_cooks"] = dds.layers["cooks"]
    out["final_robust_disp"] = robust_method_of_moments_disp(dds.layers["normed_counts"][:, nzm], dds.obsm["design_matrix"])
    out["final_mu_LFC"] = np.ascontiguousarray(dds.obsm["_mu_LFC"])
    out["final_hat"] = np.ascontiguousarray(dds.obsm["_hat_diagonals"])
    out["final_cooks_outlier"] = np.asarray(dds.cooks_outlier(), dtype=float)
    out["final_replaced"] = np.asarray(dds.var["replaced"], dtype=float)
    out["final_non_zero"] = nzm.astype(float)
    out["counts"] = counts_df.values.astype(np.int64)
    out["design"] = design_df.values.astype(float)
    out["contrast"] = np.asarray(contrast, dtype=float)
    r = pd.read_csv(r_res_csv, index_col=0)
    out["r_log2FoldChange"] = r["log2FoldChange"].values
    out["r_pvalue"] = r["pvalue"].values
    out["r_lfcSE"] = r["lfcSE"].values
    out["r_stat"] = r["stat"].values
    if r_disp_csv:
        out["r_dispersions"] = pd.read_csv(r_disp_csv, index_col=0).squeeze().values
    np.savez_compressed(os.path.join(OUT, f"tape_{name}.npz"), **out)
    # sanity: reference vs R at the reference's own tolerance (tests/test_pydeseq2.py:932-942)
    rel = np.nanmax(np.abs(r["log2FoldChange"].values - ds.results_df["log2FoldChange"].values)
                    / np.abs(r["log2FoldChange"].values))
    print(f"tape_{name}: {len(tape.calls)} calls, max rel LFC diff vs R = {rel:.2e}")


def indicator(series, level):
    return (series == level).astype(float)


def main():
    os.makedirs(OUT, exist_ok=True)
    gen_calls("two_level_n24", 24, 40, "two_level", 0)
    gen_calls("factorial_n30", 30, 40, "factorial", 1)
    gen_calls("continuous_n40", 40, 40, "continuous", 2)
    gen_calls("two_level_n200", 200, 64, "two_level", 3)
    gen_calls("large_counts_n12", 12, 40, "two_level", 4, mean_log2=18.0)
    gen_calls("five_columns_n36", 36, 40, "five", 5)
    gen_calls("intercept_n10", 10, 30, "intercept", 6)
    gen_calls("few_samples_n4", 4, 40, "two_level", 7)

    # shipped 100 x 10 synthetic dataset
    counts = pd.read_csv(f"{REF}/datasets/synthetic/test_counts.csv", index_col=0).T
    meta = pd.read_csv(f"{REF}/datasets/synthetic/test_metadata.csv", index_col=0)
    d1 = pd.DataFrame({"Intercept": 1.0, "condition[T.B]": indicator(meta["condition"], "B")}, index=meta.index)
    gen_tape("single_factor", counts, meta, d1, [0, 1], f"{REF}/tests/data/single_factor/r_test_res.csv",
             f"{REF}/tests/data/single_factor/r_test_dispersions.csv")
    d2 = pd.DataFrame({"Intercept": 1.0, "group[T.Y]": indicator(meta["group"], "Y"),
                       "condition[T.B]": indicator(meta["condition"], "B")}, index=meta.index)
    gen_tape("multi_factor", counts, meta, d2, [0, 0, 1], f"{REF}/tests/data/multi_factor/r_test_res.csv",
             f"{REF}/tests/data/multi_factor/r_test_dispersions.csv")
    # continuous covariate dataset
    cc = pd.read_csv(f"{REF}/tests/data/continuous/test_counts.csv", index_col=0).T
    cm = pd.read_csv(f"{REF}/tests/data/continuous/test_metadata.csv", index_col=0)
    print("continuous metadata columns:", list(cm.columns))
    d3 = pd.DataFrame({"Intercept": 1.0, "group[T.Y]": indicator(cm["group"], "Y"),
                       "condition[T.B]": indicator(cm["condition"], "B"),
                       "measurement": cm["measurement"].astype(float)}, index=cm.index)
    gen_tape("continuous", cc, cm, d3, [0, 0, 0, 1], f"{REF}/tests/data/continuous/r_test_res.csv")
    # wide dataset (more genes than samples)
    wc = pd.read_csv(f"{REF}/tests/data/wide/test_counts.csv", index_col=0).T
    wm = pd.read_csv(f"{REF}/tests/data/wide/test_metadata.csv", index_col=0)
    print("wide metadata columns:", list(wm.columns), wc.shape)
    d4 = pd.DataFrame({"Intercept": 1.0, "group[T.Y]": indicator(wm["group"], "Y"),
                       "condition[T.B]": indicator(wm["condition"], "B")}, index=wm.index)
    gen_tape("wide", wc, wm, d4, [0, 0, 1], f"{REF}/tests/data/wide/r_test_res.csv",
             f"{REF}/tests/data/wide/r_test_dispersions.csv")
    # outliers + a condition level with a single replicate (tests/test_pydeseq2.py:452-456): Cook's refit is triggered
    co = counts.copy()
    mo = meta.copy()
    co.loc["sample1", "gene1"] = 2000
    co.loc["sample11", "gene7"] = 1000
    mo.loc["sample1", "condition"] = "C"
    d5 = pd.DataFrame({"Intercept": 1.0, "group[T.Y]": indicator(mo["group"], "Y"),
                       "condition[T.B]": indicator(mo["condition"], "B"),
                       "condition[T.C]": indicator(mo["condition"], "C")}, index=mo.index)
    gen_tape("multi_factor_outliers", co, mo, d5, [0, 0, 1, 0], f"{REF}/tests/data/multi_factor/r_test_res_outliers.csv")

def real_fit_prior_var(lfc_col, se, coeff_idx=0):
    """The reference's own `DeseqStats._fit_prior_var` (ds.py:551-585) on bare arrays."""
    from types import SimpleNamespace

    from pydeseq2.ds import DeseqStats

    fake = SimpleNamespace(LFC=pd.DataFrame({"c": lfc_col}), SE=pd.Series(se))
    return float(DeseqStats._fit_prior_var(fake, coeff_idx=0))


def gen_shrink_calls(name, source, shrink_index, prior_scale=None):
    """apeGLM per-call fixture: the real `DefaultInference.lfc_shrink_nbinom_glm` on the inputs of an existing
    calls_* fixture (counts, design, size factors, MAP dispersions; prior scale from the MLE LFCs and Wald SEs)."""
    z = np.load(os.path.join(OUT, f"calls_{source}.npz"))
    inf = ref_inference()
    counts, X, sf, disp = z["counts"], z["X"], z["sf"], z["disp"]
    p = X.shape[1]
    contrast = np.zeros(p)
    contrast[shrink_index] = 1.0
    _, _, se = inf.wald_test(X, disp, z["lfc_beta"], np.ascontiguousarray(z["lfc_mu"]), z["ridge"], contrast, 0.0, None)
    prior_var = real_fit_prior_var(z["lfc_beta"][:, shrink_index], se)
    if prior_scale is None:
        prior_scale = float(np.minimum(np.sqrt(prior_var), 1))
    size, offset = 1.0 / disp, np.log(sf)
    lfcs, ih, conv = inf.lfc_shrink_nbinom_glm(design_matrix=X, counts=counts, size=size, offset=offset, prior_no_shrink_scale=15,
                                               prior_scale=prior_scale, optimizer="L-BFGS-B", shrink_index=shrink_index)
    np.savez_compressed(os.path.join(OUT, f"shrink_{name}.npz"), counts=counts, X=X, size=size, offset=offset, mle_lfc=z["lfc_beta"],
                        mle_se=se, prior_var=np.float64(prior_var), prior_scale=np.float64(prior_scale),
                        prior_no_shrink_scale=np.float64(15.0), shrink_index=np.int64(shrink_index), lfcs=lfcs, inv_hessians=ih,
                        converged=np.asarray(conv, dtype=float))
    print(f"shrink_{name}: G={counts.shape[1]} p={p} idx={shrink_index} prior_scale={prior_scale:.4g} converged={np.mean(conv):.3f}")


def gen_shrink_tape(name, counts_df, metadata, design_df, contrast, coeff, r_dir, r_shrunk="r_test_lfc_shrink_res.csv", adapt=True):
    """The reference's own shrinkage tests (tests/test_pydeseq2.py:256-296, 299-341, 367-430, 470-509, 566-622): R's size factors,
    dispersions, MLE LFCs and SEs go in, `lfc_shrink()` runs through the real orchestrator, R's shrunk table is stored next
    to what the reference produced."""
    from pydeseq2.dds import DeseqDataSet
    from pydeseq2.ds import DeseqStats

    r_res = pd.read_csv(f"{r_dir}/r_test_res.csv", index_col=0)
    r_shr = pd.read_csv(f"{r_dir}/{r_shrunk}", index_col=0)
    r_sf = pd.read_csv(f"{r_dir}/r_test_size_factors.csv", index_col=0).squeeze()
    r_disp = pd.read_csv(f"{r_dir}/r_test_dispersions.csv", index_col=0).squeeze()
    calls = []

    class Rec(type(ref_inference())):
        def lfc_shrink_nbinom_glm(self, **k):
            res = super().lfc_shrink_nbinom_glm(**k)
            res = (res[0], res[1], np.asarray(res[2], dtype=float))  # pandas-3: float flags (SURVEY.md §8c)
            calls.append(({kk: (np.array(v, copy=True) if hasattr(v, "shape") else v) for kk, v in k.items()}, res))
            return res

    inf = Rec(n_cpus=1)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        dds = DeseqDataSet(counts=counts_df, metadata=metadata, design=design_df, inference=inf, quiet=True)
        dds.deseq2()
        dds.obs["size_factors"] = r_sf.values
        dds.var["dispersions"] = r_disp.values
        dds.varm["LFC"].iloc[:, 1] = r_res.log2FoldChange.values * np.log(2)
        ds = DeseqStats(dds, contrast=np.asarray(contrast, dtype=float), inference=inf, quiet=True)
        ds.summary()
        ds.SE = r_res.lfcSE * np.log(2)
        coeff_idx = ds.LFC.columns.get_loc(coeff)
        mle_lfc, mle_se = ds.LFC.values.copy(), np.asarray(ds.SE, dtype=float).copy()
        prior_var = ds._fit_prior_var(coeff_idx=coeff_idx) if adapt else np.nan
        ds.lfc_shrink(coeff=coeff, adapt=adapt)
    (k, (lfcs, ih, conv)), = calls
    out = dict(counts=np.ascontiguousarray(k["counts"]).astype(np.int64), X=np.asarray(k["design_matrix"], dtype=float),
               size=np.asarray(k["size"], dtype=float), offset=np.asarray(k["offset"], dtype=float),
               prior_no_shrink_scale=np.float64(k["prior_no_shrink_scale"]), prior_scale=np.float64(k["prior_scale"]),
               shrink_index=np.int64(k["shrink_index"]), lfcs=lfcs, inv_hessians=ih, converged=np.asarray(conv, dtype=float),
               mle_lfc=mle_lfc, mle_se=mle_se, prior_var=np.float64(prior_var),
               # what ds.py:414-431 writes into LFC / SE.  Taken from the call's outputs: under pandas 3 (copy-on-write) the
               # reference's own `self.LFC.iloc[:, i].update(...)` updates a temporary and results_df keeps the MLE.
               final_log2FoldChange=lfcs[:, int(k["shrink_index"])] / np.log(2),
               final_lfcSE=np.sqrt(np.abs(ih[:, int(k["shrink_index"]), int(k["shrink_index"])])) / np.log(2),
               r_log2FoldChange=r_shr["log2FoldChange"].values, r_lfcSE=r_shr["lfcSE"].values)
    np.savez_compressed(os.path.join(OUT, f"shrinktape_{name}.npz"), **out)
    rel = np.nanmax(np.abs(out["r_log2FoldChange"] - out["final_log2FoldChange"]) / np.abs(out["r_log2FoldChange"]))
    print(f"shrinktape_{name}: G={lfcs.shape[0]} p={lfcs.shape[1]} idx={int(k['shrink_index'])} prior_scale={float(k['prior_scale']):.4g} "
          f"max rel shrunk-LFC diff vs R = {rel:.2e}")


def main_shrink():
    gen_shrink_calls("two_level_n24", "two_level_n24", 1)
    gen_shrink_calls("factorial_n30", "factorial_n30", 2)
    gen_shrink_calls("factorial_n30_idx1", "factorial_n30", 1)
    gen_shrink_calls("continuous_n40", "continuous_n40", 2)
    gen_shrink_calls("two_level_n200", "two_level_n200", 1)
    gen_shrink_calls("two_level_n200_noadapt", "two_level_n200", 1, prior_scale=1.0)
    gen_shrink_calls("large_counts_n12", "large_counts_n12", 1)
    gen_shrink_calls("five_columns_n36", "five_columns_n36", 3)
    gen_shrink_calls("few_samples_n4", "few_samples_n4", 1)
    counts = pd.read_csv(f"{REF}/datasets/synthetic/test_counts.csv", index_col=0).T
    meta = pd.read_csv(f"{REF}/datasets/synthetic/test_metadata.csv", index_col=0)
    d1 = pd.DataFrame({"Intercept": 1.0, "condition[T.B]": indicator(meta["condition"], "B")}, index=meta.index)
    gen_shrink_tape("single_factor", counts, meta, d1, [0, 1], "condition[T.B]", f"{REF}/tests/data/single_factor")
    gen_shrink_tape("single_factor_noadapt", counts, meta, d1, [0, 1], "condition[T.B]", f"{REF}/tests/data/single_factor",
                    r_shrunk="r_test_lfc_shrink_no_apeAdapt_res.csv", adapt=False)
    d2 = pd.DataFrame({"Intercept": 1.0, "group[T.Y]": indicator(meta["group"], "Y"),
                       "condition[T.B]": indicator(meta["condition"], "B")}, index=meta.index)
    gen_shrink_tape("multi_factor", counts, meta, d2, [0, 0, 1], "condition[T.B]", f"{REF}/tests/data/multi_factor")
    cc = pd.read_csv(f"{REF}/tests/data/continuous/test_counts.csv", index_col=0).T
    cm = pd.read_csv(f"{REF}/tests/data/continuous/test_metadata.csv", index_col=0)
    d3 = pd.DataFrame({"Intercept": 1.0, "group[T.Y]": indicator(cm["group"], "Y"),
                       "condition[T.B]": indicator(cm["condition"], "B"),
                       "measurement": cm["measurement"].astype(float)}, index=cm.index)
    gen_shrink_tape("continuous", cc, cm, d3, [0, 0, 0, 1], "measurement", f"{REF}/tests/data/continuous")
    lc = pd.DataFrame(data=[[25, 405, 1355, 12558, 489843], [28, 480, 2144, 13844, 514571], [12, 690, 1919, 15632, 564106],
                            [31, 420, 1684, 11513, 556380], [34, 278, 3849, 11577, 412551], [19, 249, 3086, 7296, 295565],
                            [17, 491, 4089, 13805, 280945], [15, 251, 2785, 10492, 214062]],
                      index=["A1", "A2", "A3", "A4", "B1", "B2", "B3", "B4"], columns=["g1", "g2", "g3", "g4", "g5"])
    lm = pd.DataFrame(data=["A", "A", "A", "A", "B", "B", "B", "B"], index=lc.index, columns=["condition"])
    d6 = pd.DataFrame({"Intercept": 1.0, "condition[T.B]": indicator(lm["condition"], "B")}, index=lm.index)
    gen_shrink_tape("large_counts", lc, lm, d6, [0, 1], "condition[T.B]", f"{REF}/tests/data/large_counts")


def gen_e2e(name, N, G, design_kind, seed, n_outliers, contrast_index=None, **stats_kwargs):
    """End-to-end fixture on seeded counts with injected outliers: only the final tables of the real `deseq2()` + `summary()`
    (refit of replaceable outliers, Cook's filtering of the others, independent filtering) -- the orchestration steps around
    the plugin calls (SURVEY.md §8 f-1, f-4)."""
    from pydeseq2.dds import DeseqDataSet
    from pydeseq2.ds import DeseqStats

    counts, X, _ = synth(N, G, design_kind, seed)
    rng = np.random.default_rng(seed + 100)
    for g in rng.choice(G, n_outliers, replace=False):   # one wild count per chosen gene
        counts[rng.integers(N), g] = int(counts[:, g].max() * 40 + 500)
    p = X.shape[1]
    contrast = np.zeros(p)
    contrast[p - 1 if contrast_index is None else contrast_index] = 1.0
    run_e2e(name, counts, X, contrast, **stats_kwargs)


def run_e2e(name, counts, X, contrast, r_csv=None, dds_kwargs=None, **stats_kwargs):
    from pydeseq2.dds import DeseqDataSet
    from pydeseq2.ds import DeseqStats

    N, G = counts.shape
    p = X.shape[1]
    idx = [f"s{i}" for i in range(N)]
    counts_df = pd.DataFrame(counts, index=idx, columns=[f"g{i}" for i in range(G)])
    design_df = pd.DataFrame(X, index=idx, columns=[f"x{j}" for j in range(p)])
    meta = pd.DataFrame({"dummy": np.arange(N)}, index=idx)
    inf = ref_inference()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        dds = DeseqDataSet(counts=counts_df, metadata=meta, design=design_df, inference=inf, quiet=True, **(dds_kwargs or {}))
        dds.deseq2()
        ds = DeseqStats(dds, contrast=contrast, inference=inf, quiet=True, **stats_kwargs)
        ds.summary()
    res = ds.results_df
    out = dict(counts=counts, design=X, contrast=contrast,
               final_baseMean=res["baseMean"].values, final_log2FoldChange=res["log2FoldChange"].values, final_lfcSE=res["lfcSE"].values,
               final_stat=res["stat"].values, final_pvalue=res["pvalue"].values, final_padj=res["padj"].values,
               final_LFC=dds.varm["LFC"].values, final_dispersions=dds.var["dispersions"].values,
               final_genewise=dds.var["genewise_dispersions"].values, final_fitted=dds.var["fitted_dispersions"].values,
               final_size_factors=dds.obs["size_factors"].values, final_replaced=np.asarray(dds.var["replaced"], dtype=float) if "replaced" in dds.var else np.zeros(G),
               final_refitted=np.asarray(dds.var["refitted"], dtype=float) if "refitted" in dds.var else np.zeros(G), final_cooks_outlier=np.asarray(dds.cooks_outlier(), dtype=float),
               fit_type=np.array((dds_kwargs or {}).get("fit_type", "parametric")),
               refit_cooks=np.float64((dds_kwargs or {}).get("refit_cooks", True)),
               alt_hypothesis=np.array(stats_kwargs.get("alt_hypothesis") or ""), lfc_null=np.float64(stats_kwargs.get("lfc_null", 0.0)),
               independent_filter=np.float64(stats_kwargs.get("independent_filter", True)),
               cooks_filter=np.float64(stats_kwargs.get("cooks_filter", True)), alpha=np.float64(stats_kwargs.get("alpha", 0.05)))
    if r_csv:
        r = pd.read_csv(r_csv, index_col=0)
        out.update(r_log2FoldChange=r["log2FoldChange"].values, r_stat=r["stat"].values, r_pvalue=r["pvalue"].values,
                   r_padj=r["padj"].values)
    np.savez_compressed(os.path.join(OUT, f"e2e_{name}.npz"), **out)
    print(f"e2e_{name}: N={N} G={G} p={p} replaced={int(out['final_replaced'].sum())} refitted={int(out['final_refitted'].sum())} "
          f"cooks_outlier={int(out['final_cooks_outlier'].sum())} padj<alpha={int((res['padj'] < 0.05).sum())} "
          f"padj NaN={int(res['padj'].isna().sum())} p NaN={int(res['pvalue'].isna().sum())}")


def main_e2e_edge():
    """The reference's own orchestrator-level edge cases (tests/test_edge_cases.py:323-465) on its shipped dataset."""
    counts = pd.read_csv(f"{REF}/datasets/synthetic/test_counts.csv", index_col=0).T
    meta = pd.read_csv(f"{REF}/datasets/synthetic/test_metadata.csv", index_col=0)

    def design(m):
        return np.stack([np.ones(len(m)), indicator(m["condition"], "B").values], axis=1)

    # test_few_samples: two samples per condition, one outlier -> nothing can be replaced
    keep = ["sample1", "sample2", "sample99", "sample100"]
    c = counts.loc[keep].copy()
    c.iloc[0, 0] = 1000
    run_e2e("edge_few_samples", c.values.astype(np.int64), design(meta.loc[keep]), np.array([0.0, 1.0]))
    # test_few_samples_and_outlier: a 2-sample cohort next to a 9-sample one, two outliers
    keep = ["sample1", "sample2"] + [f"sample{i}" for i in range(92, 101)]
    c = counts.loc[keep].copy()
    c.iloc[0, 0] = 1000
    c.iloc[-1, -1] = 1000
    run_e2e("edge_few_samples_and_outlier", c.values.astype(np.int64), design(meta.loc[keep]), np.array([0.0, 1.0]))
    # test_new_all_zero_gene: replacement turns geneX into an all-zero gene (and the parametric trend fit fails on 11 genes)
    keep = [f"sample{i}" for i in [*range(1, 11), *range(91, 101)]]
    c = counts.loc[keep].copy()
    c["geneX"] = 0
    c.loc["sample100", "geneX"] = 100
    run_e2e("edge_new_all_zero_gene", c.values.astype(np.int64), design(meta.loc[keep]), np.array([0.0, 1.0]))


def main_e2e_alt():
    """The reference's alternative-hypothesis test (tests/test_pydeseq2.py:180-225) on its shipped dataset, R tables alongside."""
    counts = pd.read_csv(f"{REF}/datasets/synthetic/test_counts.csv", index_col=0).T
    meta = pd.read_csv(f"{REF}/datasets/synthetic/test_metadata.csv", index_col=0)
    X = np.stack([np.ones(len(meta)), indicator(meta["condition"], "B").values], axis=1)
    for alt in ("lessAbs", "greaterAbs", "less", "greater"):
        run_e2e(f"alt_{alt}", counts.values.astype(np.int64), X, np.array([0.0, 1.0]),
                r_csv=f"{REF}/tests/data/single_factor/r_test_res_{alt}.csv",
                alt_hypothesis=alt, lfc_null=-0.5 if alt == "less" else 0.5)
    # mean-type dispersion trend (tests/test_pydeseq2.py:121-145) and no Cook's refit on data with outliers (:228-253 + :434-467)
    run_e2e("mean_fit", counts.values.astype(np.int64), X, np.array([0.0, 1.0]),
            r_csv=f"{REF}/tests/data/single_factor/r_test_res_mean_curve.csv", dds_kwargs={"fit_type": "mean"})
    co = counts.copy()
    co.loc["sample1", "gene1"] = 2000
    co.loc["sample11", "gene7"] = 1000
    run_e2e("no_refit_outliers", co.values.astype(np.int64), X, np.array([0.0, 1.0]), dds_kwargs={"refit_cooks": False})


def main_e2e():
    gen_e2e("two_level_n24", 24, 400, "two_level", 11, 12)               # cells of 12 >= 7: outliers are replaced and refitted
    gen_e2e("factorial_n20", 20, 400, "factorial", 12, 12)               # cells of 5 < 7: outliers lose their p-value instead
    gen_e2e("two_level_n16_bh", 16, 300, "two_level", 13, 8, independent_filter=False)
    gen_e2e("continuous_n30", 30, 300, "continuous", 14, 8)


def main_grid_beta():
    """``grid_beta_*.npz``: the reference's ``grid_fit_beta`` (grid_search.py:145-221) -- the last resort of ``irls_solver`` on
    two-column designs (utils.py:402-409) -- on genes of the per-call fixtures, incl. genes that are all zero in one group (the
    minimum then sits on a flat, ridge-only stretch of the grid)."""
    import pydeseq2.utils  # noqa: F401  (utils and grid_search import each other: utils first)
    from pydeseq2.grid_search import grid_fit_beta

    for source, n_genes in (("two_level_n24", 12), ("large_counts_n12", 6)):
        z = np.load(os.path.join(OUT, f"calls_{source}.npz"))
        counts, X, sf, disp = z["counts"], z["X"], z["sf"], z["disp"]
        if X.shape[1] != 2:
            continue
        counts = np.ascontiguousarray(counts[:, :n_genes])
        # two more genes: expressed in one group only / nowhere (every sample at the min_mu clamp for very negative coefficients)
        one_group = np.where(X[:, 1] > 0, counts[:, 0], 0)
        counts = np.column_stack([counts, one_group, np.zeros_like(one_group)])
        disp = np.concatenate([disp[:n_genes], [disp[0], 0.5]])
        beta = np.array([grid_fit_beta(counts[:, i], sf, X, disp[i]) for i in range(counts.shape[1])])
        np.savez_compressed(os.path.join(OUT, f"grid_beta_{source}.npz"), counts=counts, X=X, sf=sf, disp=disp, beta=beta)
        print("wrote grid_beta_" + source, beta.shape)


if __name__ == "__main__":
    from oracle import build_ref

    build_ref.build()  # the shim imports the reference package from its byte-compiled copy
    if len(sys.argv) > 1 and sys.argv[1] == "grid_beta":
        main_grid_beta()
    elif len(sys.argv) > 1 and sys.argv[1] == "e2e":  # end-to-end fixtures only
        main_e2e()
        main_e2e_edge()
        main_e2e_alt()
    elif len(sys.argv) > 1 and sys.argv[1] == "e2e_edge":
        main_e2e_edge()
    elif len(sys.argv) > 1 and sys.argv[1] == "e2e_alt":
        main_e2e_alt()
    elif len(sys.argv) > 1 and sys.argv[1] == "shrink":  # apeGLM fixtures only (reads the existing calls_* fixtures)
        main_shrink()
    else:
        main()
        main_shrink()
        main_e2e()
        main_e2e_edge()
        main_e2e_alt()
        main_grid_beta()
