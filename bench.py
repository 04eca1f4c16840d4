#!/usr/bin/env python
"""bench.py -- genes/s of the full deseq2() hot path (dispersion + IRLS + Wald) on B200, next to the CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one batch of synthetic counts: method-of-moments start values,
initial mu (lin_reg_mu or IRLS), genewise dispersion MLE, dispersion trend + prior, MAP dispersions, the
log-fold-change IRLS and the Wald test -- the Inference calls `DeseqDataSet.deseq2()` +
`DeseqStats.run_wald_test()` make (reference dds.py:516-562, ds.py:303-360) -- and, with gene shards (N > 1), the two
exchanges of the path: the per-gene vectors before the trend step and the result tables at the end of the call (one peer-memory
push kernel each, or grouped NCCL all-gathers).  Size factors are computed once outside the timed region for both arms.

Headline workload (`value`, `e2e`, `roofline`, `cpu_baseline`) = BASELINE.json configs[1]: 20 000 genes x 200 samples, one
2-level factor, per GPU (weak scaling).  The `configs` block of the same JSON line carries BASELINE's larger shapes, timed the
same way: C3 (60 000 x 500, 3 covariates, one GPU holds it) at N = 1, and at every N the per-GPU shards of the two 8-GPU
configs, C5 (125 000 x 1 000 of 10^6 x 1 000) and C4 (7 500 x 2 000 of 60 000 x 2 000, continuous covariate).

Prints ONE JSON line (rank 0).  `value` = device-resident throughput (counts already in HBM), timed per step with
CUDA events on the library's stream, L2 flushed between steps, max over ranks.  `e2e` = the same metric through the
reference-facing plugin calls with HOST buffers (H2D/D2H inside the timed region; page-locked and pageable variants).
`roofline` describes the dominant kernel, `cpu_baseline` the oracle port (joblib over genes, like the reference).

Every timed loop on the device runs exactly K steps, as does the reference arm; the device arm's `cpu_baseline` is a fixed
three passes.  `--dump-outputs DIR` writes what the last timed step of the headline workload returned (rank 0's shard) as
DIR/<name>.npy in float64; the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "genes/sec full deseq2() fit (disp+IRLS+Wald)"
UNIT = "genes/s"
P_OF = {"two_level": 2, "factorial": 3, "continuous": 3}
# bytes per (gene, sample) each Inference call reads + writes once: SURVEY.md §8(d)
ALG_BYTES = {"mom_dispersions": 8, "lin_reg_mu": 16, "irls_init": 24, "alpha_mle_genewise": 16, "alpha_mle_map": 16,
             "irls_lfc": 24, "irls_lfc_wald": 24, "wald_test": 8}
KERNEL_OF = {"alpha_mle_genewise": "k_alpha_mle", "alpha_mle_map": "k_alpha_mle", "irls_lfc": "k_irls", "irls_lfc_wald": "k_irls",
             "irls_init": "k_irls", "lin_reg_mu": "k_lin_reg_mu", "wald_test": "k_wald", "mom_dispersions": "k_mom_from_counts"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of every device measurement and of the reference arm (cpu_baseline: a fixed 3 passes)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--genes", type=int, default=20000)
    ap.add_argument("--samples", type=int, default=200)
    ap.add_argument("--design", default="two_level", choices=["two_level", "factorial", "continuous"])
    ap.add_argument("--cpu-sample-genes", type=int, default=20000,
                    help="genes of the workload the CPU baseline is timed on (20 000 x 200 is ~6 s per pass on the GPU box)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-configs", action="store_true", help="skip the `configs` block (C3 / C5 shard / C4 shard)")
    ap.add_argument("--lanes", type=int, default=0, help="lanes per gene override (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the arrays the last timed step of the headline workload returned as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(out_dir, res, limit=64 << 20):
    """The per-gene tables and trend record one pass of `ResidentFit.run` hands its caller, as float64 .npy files (a few MB at the
    headline workload).  Above `limit` bytes the per-gene tables keep a fixed, seeded sample of genes, listed in gene_index.npy."""
    scalars = {"prior_var": res["prior_var"], "squared_logres": res["squared_logres"], "trend_coeffs": res["trend"].coeffs}
    per_gene = {k: np.asarray(v, dtype=np.float64) for k, v in res.items() if k not in scalars and k != "trend"}
    G = len(res["dispersions"])
    row_bytes = sum(a.nbytes for a in per_gene.values()) // max(G, 1)
    if G * row_bytes > limit:
        keep = (limit - (1 << 16)) // (row_bytes + 8)  # + gene_index, and room for the .npy headers and the scalars
        idx = np.sort(np.random.default_rng(0).choice(G, keep, replace=False))
        per_gene = {k: a[idx] for k, a in per_gene.items()}
        per_gene["gene_index"] = idx.astype(np.float64)
    arrays = {**per_gene, **{k: np.atleast_1d(np.asarray(v, dtype=np.float64)) for k, v in scalars.items()}}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def make_workload(samples, genes, design, rank, dist=None):
    """This rank's gene shard of one synthetic cohort: samples (design matrix, true size factors) are common to all ranks, genes
    are drawn per rank; the median-of-ratios size factors are per sample and global over genes -- rank 0's estimate serves all."""
    from pydeseq2_b200.pipeline import median_of_ratios
    from pydeseq2_b200.synth import make_counts

    counts, X, _ = make_counts(samples, genes, design, seed=rank, sample_seed=0)
    G_in = counts.shape[1]
    counts = np.ascontiguousarray(counts[:, ~(counts == 0).all(0)])  # dds.py:729-731 (throughput counts input G)
    _, sf = median_of_ratios(counts[:, :20000])
    if dist is not None:
        import torch

        t = torch.from_numpy(sf).cuda()
        dist.broadcast(t, 0)
        sf = t.cpu().numpy()
    return counts, X, sf, G_in


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, STREAM-style copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def profile_record():
    path = os.path.join(ROOT, "profiles", "traffic.json")
    return json.load(open(path)) if os.path.exists(path) else {}


def cpu_fit(counts, X, sf, n_cpus):
    """The reference CPU path (oracle port: numpy/scipy per gene, joblib/loky over genes)."""
    from oracle import nbglm  # the one place bench.py may execute oracle/: the CPU baseline
    from pydeseq2_b200.pipeline import fit_host

    inf = nbglm.OracleInference(n_cpus=n_cpus)
    t0 = time.perf_counter()
    fit_host(counts, X, inf, size_factors=sf)
    return time.perf_counter() - t0


def cpu_sample_desc(n, args, passes):
    return (f"{'all' if n >= args.genes else 'first'} {n} of {args.genes} genes x {args.samples} samples "
            f"(non-all-zero genes of them), median of {passes} timed passes after a warm-up pass")


def run_reference(args, rank, world):
    """CPU arm: the oracle port of DefaultInference on all host cores, the FULL headline workload per step."""
    if rank != 0:
        return
    counts, X, sf, G_in = make_workload(args.samples, args.genes, args.design, 0)
    n_in = min(args.cpu_sample_genes, G_in)
    sample = counts if n_in >= G_in else np.ascontiguousarray(counts[:, :n_in])
    cores = os.cpu_count() or 1
    cpu_fit(sample[:, :256], X, sf, cores)  # spawn the loky pool outside the timed region
    for _ in range(max(1, min(args.warmup, 2))):
        cpu_fit(sample, X, sf, cores)
    steps = args.steps
    times = [cpu_fit(sample, X, sf, cores) for _ in range(steps)]
    dt = float(np.median(times))
    val = n_in / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": max(1, min(args.warmup, 2)), "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config(args, note=f"reference CPU path: oracle port of DefaultInference (numpy/scipy per gene, joblib/loky, "
                                        f"{cores} processes); each step = {cpu_sample_desc(n_in, args, steps)}"),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": cpu_sample_desc(n_in, args, steps),
                             "pass_s": [round(t, 3) for t in times]},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def config(args, note=None):
    p = P_OF[args.design]
    c = {"workload": f"{args.genes} genes x {args.samples} samples per GPU, {args.design} design (p={p}); BASELINE.json configs[1]"
                     if (args.genes, args.samples, args.design) == (20000, 200, "two_level")
                     else f"{args.genes} genes x {args.samples} samples per GPU, {args.design} design (p={p})",
         "genes_per_gpu": args.genes, "samples": args.samples, "p": p,
         "parallelism": f"gene shards x{args.gpus}; per step one exchange of the per-gene vectors before the trend fit and one of the "
                        f"result tables at the end (one push kernel each over peer memory / NVLink; grouped NCCL all-gathers when the "
                        f"ranks cannot map each other's memory -- see `exchange`)",
         "size_factors": "median of ratios, precomputed outside the timed region (both arms)",
         "l2": "flushed between timed steps (256 MiB device memset)"}
    if note:
        c["note"] = note
    return c


class Bench:
    """One process = one GPU: context, NCCL communicator (N > 1) and the measurements of one workload at a time."""

    def __init__(self, args):
        self.args = args
        self.rank = int(os.environ.get("RANK", 0))
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.local = int(os.environ.get("LOCAL_RANK", 0))
        self.dist = None
        if self.world > 1:
            import torch
            import torch.distributed as dist

            torch.cuda.set_device(self.local)
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
        from pydeseq2_b200 import _lib
        from pydeseq2_b200.inference import B200Inference

        self._lib = _lib
        self.inf = B200Inference(device=self.local, lanes_per_gene=args.lanes)
        self.ctx = self.inf._ops.ctx
        self.uid = None
        if self.world > 1:
            import torch
            from pydeseq2_b200.sharding import NcclComm

            uid = torch.zeros(_lib.UNIQUE_ID_BYTES, dtype=torch.uint8, device="cuda")
            if self.rank == 0:
                uid.copy_(torch.frombuffer(bytearray(NcclComm.make_unique_id(self.ctx)), dtype=torch.uint8))
            self.dist.broadcast(uid, 0)
            self.uid = uid.cpu().numpy().tobytes()
        self.comm = None
        self.flush = self.ctx.malloc(256 << 20)
        self.peak, self.peak_src = peaks()
        self.fp64_peak = None

    # -- plumbing ---------------------------------------------------------------------------------------------
    def barrier(self):
        self.ctx.sync()
        if self.dist is not None:
            import torch

            self.dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(self, v):
        if self.dist is None:
            return float(v)
        import torch

        t = torch.tensor([float(v)], device="cuda", dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def all_sizes(self, G):
        if self.dist is None:
            return [G]
        import torch

        t = torch.tensor([G], device="cuda", dtype=torch.int64)
        out = [torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [int(o.item()) for o in out]

    def comm_for(self, G):
        """Shard sizes differ per workload (every rank drops its own all-zero genes): one NCCL communicator, sizes re-set."""
        if self.world == 1:
            return None
        from pydeseq2_b200.sharding import NcclComm

        sizes = self.all_sizes(G)
        if self.comm is None:
            self.comm = NcclComm(self.ctx, sizes, self.rank, self.uid)
        else:
            self.comm.sizes, self.comm.max_size = list(sizes), max(sizes)
        return self.comm

    def flush_l2(self):
        self.ctx.check(self.ctx.lib.pdq_memset(self.ctx.h, self._lib.c_dptr(self.flush), 1, 256 << 20))
        self.ctx.sync()

    # -- measurements -----------------------------------------------------------------------------------------
    def resident(self, counts, X, sf, G_in, steps, warmup, exchange=None):
        """Device-resident steps (CUDA events on the library's stream, L2 flushed, max over ranks) + per-stage timings."""
        from pydeseq2_b200.pipeline import ResidentFit

        N, G = counts.shape
        rf = ResidentFit(self.ctx, X, sf, comm=self.comm_for(G))
        if exchange:
            rf.exchange = exchange
        rf.upload(counts)
        for _ in range(max(warmup, 3)):
            rf.run()
        self.barrier()
        launches0 = self.ctx.launches()
        step_ms = []
        for _ in range(steps):
            self.flush_l2()
            self.barrier()
            out = rf.run(events=(0, 1))  # CUDA events around the device work of the pass: first launch ... result copy done
            step_ms.append(self.ctx.elapsed_ms(0, 1))
        self.barrier()
        launches = self.ctx.launches() - launches0
        ms = self.max_over_ranks(float(np.sum(step_ms))) / steps
        rf.run(profile=True)
        rf.run(profile=True)
        stages = dict(rf.stage_ms)
        rec = {"ms_per_step": ms, "genes_per_s": G_in * self.world / (ms * 1e-3), "gpu_launches": int(launches),
               "stages_ms": {k: round(v, 4) for k, v in stages.items()}}
        if self.world > 1:  # how the shards exchanged: peer-memory push kernel (NVLink stores) or grouped NCCL all-gathers
            rec["exchange"] = "peer" if rf._win is not None else "nccl"
        rec.update(self.rooflines(stages, N, G, X.shape[1], ms))
        return rf, rec, out

    def rooflines(self, stages, N, G, p, step_ms):
        """HBM roofline of the dominant kernel and of the whole step; FP64 roofline of the dominant kernel (DFMA peak measured in
        this run; flop count per (gene, sample) from the committed ncu capture of the same kernel, profiles/traffic.json)."""
        kern = {k: v for k, v in stages.items() if k in ALG_BYTES}
        top = max(kern, key=kern.get)
        achieved = ALG_BYTES[top] * N * G / (kern[top] * 1e-3) / 1e9
        step_bytes = sum(ALG_BYTES[k] for k in kern) * N * G
        if "irls_lfc_wald" in kern:
            step_bytes += ALG_BYTES["wald_test"] * N * G  # the fused launch also does the Wald call's work (its mu read is saved)
        kname = KERNEL_OF[top]
        prof = profile_record()
        roof = {"bound": "hbm", "kernel": f"{kname} ({top})", "achieved": achieved, "peak": self.peak, "unit": "GB/s",
                "frac": achieved / self.peak, "traffic": prof.get("dram_bytes_per_launch", {}).get(kname),
                "peak_source": self.peak_src, "algorithmic_bytes_per_launch": ALG_BYTES[top] * N * G, "kernel_ms": kern[top],
                "step": {"algorithmic_bytes": step_bytes, "achieved": step_bytes / (step_ms * 1e-3) / 1e9,
                         "frac": step_bytes / (step_ms * 1e-3) / 1e9 / self.peak},
                "note": "issue / FP64-pipe bound (log, exp, reciprocal, digamma per gene-sample-iteration), see DESIGN.md §5"}
        if self.fp64_peak is None:
            self.fp64_peak = self.ctx.fp64_peak_tflops()
        fp64 = {"peak_tflops": self.fp64_peak, "peak_source": "measured in this run (pdq_fp64_peak_tflops: DFMA chains on every SM)"}
        by_n = prof.get("fp64_flop_per_gene_sample_by_samples", {})
        if by_n:  # counters exist for the captured sample counts (200, 500): take the nearest
            key = min(by_n, key=lambda k: abs(int(k) - N))
            per_pair = by_n[key].get(kname)
            fp64["flop_counted_at_samples"] = int(key)
        else:
            per_pair = prof.get("fp64_flop_per_gene_sample", {}).get(kname)
        if per_pair:
            flop = per_pair * N * G
            fp64.update({"achieved_tflops": flop / (kern[top] * 1e-3) / 1e12, "flop_per_launch": flop,
                         "frac": flop / (kern[top] * 1e-3) / 1e12 / self.fp64_peak if self.fp64_peak > 0 else None,
                         "flop_source": prof.get("fp64_flop_source"),
                         "pipe_active_pct_ncu": prof.get("fp64_pipe_active_pct", {}).get(kname)})
        roof["fp64"] = fp64
        return {"roofline": roof}

    def e2e(self, counts, X, sf, G_in, steps, pinned):
        """The same pass through the plugin calls with HOST buffers (H2D / D2H inside the timed region).  `pinned`: the caller's
        (N, G) inputs are page-locked and handed on as they are (best case).  Not `pinned`: what the reference's orchestrator
        does -- pageable inputs, and every call receives a FRESH pageable copy of its (N, G) arguments (dds.py:752, 759, 779,
        902, 954); the copies are the orchestrator's work and are subtracted from the step (reported alongside)."""
        from pydeseq2_b200.pipeline import fit_host

        inf = self.inf
        alloc = (lambda shape, dt: self.ctx.pinned_empty(shape, dt)) if pinned else (lambda shape, dt: np.empty(shape, dt))
        c_host = alloc(counts.shape, np.int64)
        c_host[:] = counts
        n_host = alloc(counts.shape, np.float64)  # layers["normed_counts"] of the orchestrator (dds.py:700-708)
        np.divide(counts, sf[:, None], out=n_host)
        n_means = n_host.mean(0)  # var["_normed_means"], also a product of fit_size_factors (dds.py:708)
        comm = self.comm_for(counts.shape[1])
        kw = dict(size_factors=sf, comm=comm, normed_counts=n_host, normed_means=n_means, fresh_copies=not pinned)
        for _ in range(2):
            fit_host(c_host, X, inf, **kw)
        self.barrier()
        ops = inf._ops
        h0, d0 = ops.h2d_bytes, ops.d2h_bytes
        stats0 = self.ctx.residency_stats()
        ts, T = [], {}
        for _ in range(steps):
            self.barrier()
            t0 = time.perf_counter()
            fit_host(c_host, X, inf, timings=T, **kw)
            ops.ctx.sync()
            ts.append(time.perf_counter() - t0)
        copies = T.pop("orchestrator_copies", 0.0) / steps
        in_calls = sum(T.values()) / steps  # wall time spent INSIDE the plugin calls (+ the all-gather of gene shards)
        # page-locked variant: the whole step's wall clock.  Pageable variant: the time inside the plugin calls -- the rest of that
        # step is the orchestrator making and releasing its fresh 32 MB copies (mmap / munmap, page faults), which is not backend work
        s = self.max_over_ranks(float(np.mean(ts)) if pinned else in_calls)
        stats1 = self.ctx.residency_stats()
        return {"value": G_in * self.world / s, "unit": UNIT, "ms_per_step": s * 1e3,
                "h2d_bytes_per_step": (ops.h2d_bytes - h0) // steps - (stats1["hit_bytes"] - stats0["hit_bytes"]) // steps,
                "d2h_bytes_per_step": (ops.d2h_bytes - d0) // steps,
                "h2d_bytes_skipped_resident_per_step": (stats1["hit_bytes"] - stats0["hit_bytes"]) // steps,
                "host_buffers": "page-locked inputs, passed on unchanged" if pinned else
                                "pageable inputs, a fresh pageable copy per plugin call (the orchestrator's fancy-indexed copies, dds.py:752)",
                "timed": "wall clock of the step" if pinned else "wall clock inside the plugin calls of the step",
                "in_calls_ms": round(in_calls * 1e3, 3), "orchestrator_copies_ms": round(copies * 1e3, 3),
                "step_wall_ms": [round(t * 1e3, 2) for t in ts],
                "calls_ms": {k: round(v * 1e3 / steps, 3) for k, v in T.items()}}

    def full_deseq2(self, counts, X, sf, G_in, steps):
        """Second metric (N = 1): the whole `DeseqDataSet.deseq2()` of the reference (dds.py:516-562) -- the hot path PLUS
        `calculate_cooks` and the outlier `refit` -- and the Wald test, resident: one pass with Cook's distances on the device,
        then the replaced genes' refit on a compact resident matrix (workflow.deseq2_results_resident).  Wall clock per call."""
        from pydeseq2_b200.pipeline import ResidentFit
        from pydeseq2_b200.workflow import deseq2_results_resident

        rf = ResidentFit(self.ctx, X, sf)
        rf.upload(counts)
        for _ in range(2):
            r = deseq2_results_resident(rf, adjust=False)
        ts = []
        for _ in range(steps):
            self.flush_l2()
            t0 = time.perf_counter()
            r = deseq2_results_resident(rf, adjust=False)
            ts.append(time.perf_counter() - t0)
        rf.close()
        s = float(np.mean(ts))
        return {"metric": "genes/sec deseq2() incl. Cook's distances + outlier refit, + Wald", "ms_per_step": s * 1e3, "genes_per_s": G_in / s,
                "timed": "wall clock per call (counts resident; includes the host-side replacement of the flagged genes' counts)",
                "replaced_genes": int(r.replaced.sum()), "refitted_genes": int(r.refitted.sum()),
                "cooks_outlier_genes": int(r.cooks_outlier.sum())}

    def check_shards(self, rf):
        """N > 1: the sharded pass must equal a single-process fit -- (a) every rank holds the same trend record and tables,
        (b) the trend / prior of the gathered vectors recomputed by ONE rank on the concatenation (no NaN pads) agree."""
        import torch

        res = rf.run()
        full = rf.gather_results(res)
        t16 = torch.from_numpy(np.array([res["trend"].coeffs[0], res["trend"].coeffs[1], res["prior_var"], res["squared_logres"],
                                         float(np.nansum(full["dispersions"])), float(np.nansum(np.abs(full["lfc"]))),
                                         float(len(full["dispersions"]))])).cuda()
        outs = [torch.empty_like(t16) for _ in range(self.world)]
        self.dist.all_gather(outs, t16)
        same = all(bool(torch.equal(o, outs[0])) for o in outs)
        out = {"ranks_hold_identical_tables": same, "genes_gathered": int(len(full["dispersions"]))}
        if self.rank == 0:
            tp = self.inf.trend_and_prior(full["normed_means"], full["genewise"], rf.min_disp, rf.max_disp, rf.N, rf.p)
            if tp is not None:
                out["trend_coeff_rel_err_vs_single_process"] = float(np.max(np.abs(tp[0] / res["trend"].coeffs - 1)))
                out["prior_var_rel_err_vs_single_process"] = abs(tp[3] / res["prior_var"] - 1)
                out["ok"] = bool(same and out["trend_coeff_rel_err_vs_single_process"] < 1e-9
                                 and out["prior_var_rel_err_vs_single_process"] < 1e-9)
        return out


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args, int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)))
    B = Bench(args)
    rank, world, ctx = B.rank, B.world, B.ctx
    counts, X, sf, G_in = make_workload(args.samples, args.genes, args.design, rank, B.dist)
    N, G = counts.shape

    # ---------------------------------------------------------------- value: device-resident (headline workload)
    clk = ClockSampler(B.local).__enter__()  # sampled from the warm-up until the end of the e2e loop (steps last only ms)
    rf, head, last_out = B.resident(counts, X, sf, G_in, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_out)
    stages = dict(head["stages_ms"])
    shard_check = B.check_shards(rf) if world > 1 else None
    exchange_ab = None
    if world > 1 and head.get("exchange") == "peer":  # the same steps with the NCCL exchange, for comparison
        rf_n, rec_n, _ = B.resident(counts, X, sf, G_in, args.steps, args.warmup, exchange="nccl")
        rf_n.close()
        exchange_ab = {"peer_ms_per_step": head["ms_per_step"], "nccl_ms_per_step": rec_n["ms_per_step"],
                       "nccl_stages_ms": {k: rec_n["stages_ms"][k] for k in ("allgather", "gather_results") if k in rec_n["stages_ms"]}}

    # untimed extras (reported for information, NOT part of the timed step): Cook's distances, apeGLM shrinkage, device size factors
    from pydeseq2_b200.pipeline import fit_shrink_prior_var

    rf.with_cooks = True
    rf.run(profile=True)
    stages["cooks_untimed"] = round(rf.stage_ms.get("cooks", float("nan")), 4)
    rf.with_cooks = False
    res_sh = rf.run()
    k_sh = X.shape[1] - 1
    ps_sh = float(min(np.sqrt(fit_shrink_prior_var(np.asarray(res_sh["lfc"])[:, k_sh], np.asarray(res_sh["se"]))), 1.0))
    rf.lfc_shrink(res_sh, k_sh, prior_scale=ps_sh)  # first call allocates its buffers
    t0 = time.perf_counter()
    rf.lfc_shrink(res_sh, k_sh, prior_scale=ps_sh)
    stages["lfc_shrink_untimed"] = round((time.perf_counter() - t0) * 1e3, 4)
    if world == 1:
        rf.device_size_factors()  # first call allocates its scratch
        ctx.sync()
        t0 = time.perf_counter()
        rf.device_size_factors()
        stages["size_factors_dev_untimed"] = round((time.perf_counter() - t0) * 1e3, 4)
    rf.close()

    # ---------------------------------------------------------------- e2e: plugin calls with host buffers
    e2e = B.e2e(counts, X, sf, G_in, args.steps, pinned=True)
    e2e_pageable = B.e2e(counts, X, sf, G_in, args.steps, pinned=False)
    e2e["pageable"] = e2e_pageable
    time.sleep(0.25)  # let nvidia-smi emit at least one more sample
    clk.__exit__()

    full = B.full_deseq2(counts, X, sf, G_in, args.steps) if world == 1 else None

    # ---------------------------------------------------------------- BASELINE's larger shapes, same measurement
    configs = {}
    if not args.no_extra_configs and (args.genes, args.samples, args.design) == (20000, 200, "two_level"):
        extra = [("C5_shard", 125000, 1000, "two_level", "BASELINE.json configs[4] (10^6 x 1 000 over 8 GPUs): one 125 000-gene shard per GPU"),
                 ("C4_shard", 7500, 2000, "continuous", "BASELINE.json configs[3] (60 000 x 2 000 over 8 GPUs): one 7 500-gene shard per GPU")]
        if world == 1:
            extra.insert(0, ("C3", 60000, 500, "factorial", "BASELINE.json configs[2]: 60 000 genes x 500 samples, 3 covariates, whole on one GPU"))
        for name, g, n, design, what in extra:
            c2, X2, sf2, gin2 = make_workload(n, g, design, rank, B.dist)
            rf2, rec, _ = B.resident(c2, X2, sf2, gin2, args.steps, 3)
            rec["workload"] = f"{what}; {g} genes x {n} samples per GPU, {design} design (p={P_OF[design]})"
            if world > 1:
                rec["shard_check"] = B.check_shards(rf2)
            rf2.close()
            if name == "C3":
                rec["e2e"] = B.e2e(c2, X2, sf2, gin2, args.steps, pinned=True)
            configs[name] = rec
            del c2, rf2

    # ---------------------------------------------------------------- CPU baseline (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n_in = min(args.cpu_sample_genes, G_in)
        cores = os.cpu_count() or 1
        sample = counts if n_in >= G_in else np.ascontiguousarray(counts[:, :n_in])
        cpu_fit(sample[:, :256], X, sf, cores)  # pool start-up outside the timed region
        cpu_fit(sample, X, sf, cores)           # warm-up pass
        times = [cpu_fit(sample, X, sf, cores) for _ in range(3)]
        dt = float(np.median(times))
        cpu = {"value": n_in / dt, "unit": UNIT, "cores": cores, "kind": "port", "sample": cpu_sample_desc(n_in, args, 3),
               "pass_s": [round(t, 3) for t in times]}

    if rank == 0:
        line = {"metric": METRIC, "value": head["genes_per_s"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config(args), "e2e": e2e,
                "gpu_launches": head["gpu_launches"], "clocks": clk.summary(), "roofline": head["roofline"], "cpu_baseline": cpu,
                "stages_ms": stages, "full_deseq2": full, "configs": configs, "shard_check": shard_check, "exchange": head.get("exchange"), "exchange_ab": exchange_ab,
                "device": ctx.info()["name"]}
        print(json.dumps(line), flush=True)
    if B.dist is not None:
        B.dist.barrier()
        B.dist.destroy_process_group()


if __name__ == "__main__":
    main()
