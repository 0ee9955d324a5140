#!/usr/bin/env python
"""Cost of projecting held-out samples (vpca_create_projecting) at the size of the 1000 Genomes panel: N = 2504 fitted
samples, M in {0, 256, 2504} projected ones, 1 M synthetic variants held in HBM in panel layout (int8, binary carriers).

For every M, on one GPU:
  * the Gram launch (fitted lower triangle + M x N cross block) from CUDA events after warm-up, over enough launches to
    fill >= 1 s; executed operations (N (N + 1) + 2 M N) V and the rate;
  * vpca_compute_pca (device time of centring + eigensolve, vpca_stats.last_eig_ms) and the projection kernels
    (torch.profiler, CUDA activity of the proj_* kernels, in a pass of its own);
  * checks: the fitted block bit for bit against a plain context fed the same N fitted rows, and sampled cross rows
    exactly against an fp32 matmul of the same genotypes (0/1 cells, counts < 2^24, TF32 off).
M = 0 also runs through vpca_create_projecting and is timed against a plain vpca_create context, launches alternating:
the tile list is the same, so the times should be.  The device name and power limit are read (read-only) in the same run."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np
import torch
from spark_examples_b200 import native

SEED = 20240901


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def time_launches(runs, min_s, min_launches=5):
    """runs: list of (name, fn) enqueuing one launch each; alternated until each has >= min_s of device time."""
    ms = {name: [] for name, _ in runs}
    while min(sum(v) for v in ms.values()) < 1e3 * min_s or min(len(v) for v in ms.values()) < min_launches:
        for name, fn in runs:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ms[name].append(a.elapsed_time(b))
    return {name: {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "launches": len(v)} for name, v in ms.items()}


def panel_rows(buf, rows_total, P, rows, nv):
    """fp32 (len(rows), nv) copy of the given rows of a panel buffer"""
    v = buf.view(-1, rows_total, P)[:, rows, :]                  # (panels, r, P)
    return v.permute(1, 0, 2).reshape(len(rows), -1)[:, :nv].float()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--projected", default="0,256,2504")
    ap.add_argument("--variants", type=int, default=1_000_000)
    ap.add_argument("--panel", type=int, default=8192)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--check-rows", type=int, default=8)
    ap.add_argument("--k", type=int, default=2)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("project_bench.py measures on the GPU: no CUDA device")
    n, nv, P, k = args.samples, args.variants, args.panel, args.k
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    report = dict(device_info(), samples=n, variants=nv, panel=P, dtype="int8", k=k, results=[])
    all_ok = True
    torch.backends.cuda.matmul.allow_tf32 = False
    for m in [int(x) for x in args.projected.split(",")]:
        total = n + m
        rows_map = np.arange(total, dtype=np.int32)                      # M = 0 still goes through vpca_create_projecting
        proj = native.NativePca(n, stream=stream.cuda_stream, max_multiplicity=1, n_projected=m, sample_rows=rows_map)
        buf = torch.zeros(proj.panelBytes(nv, P), dtype=torch.uint8, device="cuda")
        proj.synthPanelsDevice(SEED, 0, nv, 0, buf.data_ptr(), P)
        # the fitted rows alone, for a plain context: rows [0, N) of every panel
        fit_buf = buf.view(-1, total, P)[:, :n, :].contiguous().view(-1)
        plain = native.NativePca(n, stream=stream.cuda_stream, max_multiplicity=1)

        def run(ctx, b):
            def f():
                ctx.reset()
                ctx.accumulatePanels(b.data_ptr(), nv, P)
            return f
        runs = [("projecting", run(proj, buf))] + ([("plain", run(plain, fit_buf))] if m == 0 else [])
        for _ in range(3):                                               # warm-up (module load, adaptive split)
            for _, fn in runs:
                fn()
        stream.synchronize()
        times = time_launches(runs, args.min_seconds)
        ops = float(n * (n + 1) + 2 * m * n) * nv                         # executed MACs x 2 of the lower triangle + cross
        res = {"n_projected": m, "tiles": int(len(native.debugProjectionTiles(n, total, 2, False))),
               "gram": times["projecting"], "ops": ops,
               "tops": ops / (times["projecting"]["median_ms"] * 1e-3) / 1e12,
               "gram_resident": proj.stats()["gram_resident"]}
        if m == 0:
            res["plain_gram"] = times["plain"]
        # ---- fitted block + cross block, checked
        proj.reset()
        proj.accumulatePanels(buf.data_ptr(), nv, P)
        proj.finalizeGram()
        plain.reset()
        plain.accumulatePanels(fit_buf.data_ptr(), nv, P)
        plain.finalizeGram()
        fitted_ok = bool(np.array_equal(proj.getGram(), plain.getGram()))
        cross_ok = True
        if m > 0:
            X = proj.crossGram()
            rng = np.random.default_rng(m)
            sample = sorted(set([0, m - 1] + rng.choice(m, size=min(m, args.check_rows), replace=False).tolist()))
            xp = panel_rows(buf, total, P, [n + p for p in sample], nv)
            want = torch.zeros((len(sample), n), dtype=torch.float32, device="cuda")
            for f0 in range(0, n, 512):                                   # fitted rows in slabs: bounded fp32 memory
                f1 = min(n, f0 + 512)
                want[:, f0:f1] = xp @ panel_rows(buf, total, P, list(range(f0, f1)), nv).T
            cross_ok = bool(np.array_equal(X[sample], want.to(torch.int32).cpu().numpy()))
            res["cross_rows_checked"] = len(sample)
        # ---- compute_pca, projection
        eig = []
        for _ in range(5):
            proj.computePca(k)
            eig.append(proj.stats()["last_eig_ms"])
        res["compute_pca_ms_median"] = float(np.median(eig[1:]))
        res["eig_method"] = proj.stats()["eig_method"]
        vecs, evals, _ = proj.computePca(k)
        pv, pe, _ = plain.computePca(k)
        pca_ok = bool(np.array_equal(vecs, pv) and np.array_equal(evals, pe))
        if m > 0:
            y = proj.projectPca(k)
            repeat_ok = bool(np.array_equal(y, proj.projectPca(k)))
            t0 = time.perf_counter()
            reps = 50
            for _ in range(reps):
                proj.projectPca(k)
            res["project_call_ms_host"] = (time.perf_counter() - t0) * 1e3 / reps
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for _ in range(10):
                    proj.projectPca(k)
            kern = {}
            for e in prof.key_averages():
                for name in ("proj_rowmean", "proj_dot", "proj_finish"):
                    if name in e.key:
                        t = getattr(e, "device_time_total", None)
                        kern[name] = kern.get(name, 0.0) + (t if t is not None else e.cuda_time_total) / 10.0
            res["project_kernels_us"] = {kk: round(v, 2) for kk, v in kern.items()}
            res["project_kernels_us_total"] = round(sum(kern.values()), 2)
            res["project_algorithmic_bytes"] = 4 * m * n + 8 * n * k + 8 * m * k
            res["project_repeat_bit_identical"] = repeat_ok
            pca_ok = pca_ok and repeat_ok
        res["checks"] = {"fitted_block_equals_plain": fitted_ok, "cross_rows_exact": cross_ok,
                         "pca_equals_plain_and_repeatable": pca_ok}
        all_ok = all_ok and fitted_ok and cross_ok and pca_ok
        report["results"].append(res)
        print(json.dumps(res), flush=True)
        proj.close()
        plain.close()
        del buf, fit_buf
        torch.cuda.empty_cache()
    report["all_checks_pass"] = all_ok
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(report, indent=1) + "\n")
    print(json.dumps({"all_checks_pass": all_ok}))
    if not all_ok:
        raise SystemExit(1)


if __name__ == "__main__":
    main()
