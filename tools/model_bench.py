#!/usr/bin/env python
"""Cost of the saved-model passes (DESIGN.md 3.7) at the size of the 1000 Genomes panel: N = 2504 fitted samples and
1 M synthetic int8 variants (binary carriers) held in HBM in panel layout.

On one GPU, in one run:
  * the loadings pass (vpca_pca_loadings_panels) for k = 2 and k = 16;
  * the scoring pass (vpca_score_panels) of M in {256, 2504} study samples for k = 2;
  * the current way to get the same coordinates at the same M: the vpca_create_projecting Gram launch and vpca_project_pca.
Kernel times are the device durations of the model_* kernels (torch.profiler, CUDA activity) summed over >= 1 s of kernel
time after warm-up; the Gram launch is timed with CUDA events like tools/project_bench.py.  For each pass the tool computes
from shapes the algorithmic bytes (cells read once, loadings / partials) and FP64 operations (one FMA per cell and column),
the HBM bound (7.7 TB/s) and the FP64 bound (37 TFLOP/s, the data-sheet FP64 rate of one HGX B200 GPU), and says which one is
larger.  Checks: loadings of k = 2 equal the first two columns of k = 16 bit for bit and agree with an FP64 X^T U of sampled
variants; the scores of every M agree with vpca_project_pca of the same panel and study to 1e-9 x max|y_c|; the first
256 fitted samples scored as a study land on their fitted coordinates to 1e-9; repeated scoring is bit-identical.  The
device name, power limit and max SM clock are read (read-only) in the same run."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np
import torch
from spark_examples_b200 import native

SEED = 20240901
HBM_BYTES_PER_S = 7.7e12
FP64_FLOPS = 37e12


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def kernel_ms(fn, names, min_s):
    """Device time per call of the kernels whose name contains one of `names`, summed over >= min_s of it."""
    def profiled(reps):
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                fn()
            torch.cuda.synchronize()
        tot = 0.0
        for e in prof.key_averages():
            if any(nm in e.key for nm in names):
                t = getattr(e, "device_time_total", None)
                tot += t if t is not None else e.cuda_time_total
        return tot / 1e3   # ms
    for _ in range(3):
        fn()                                    # warm-up
    probe = profiled(3) / 3
    reps = max(5, int(np.ceil(1e3 * min_s / max(probe, 1e-3))))
    total = profiled(reps)
    return total / reps, reps, total


def bound(bytes_, flops, ms):
    hbm, fp = bytes_ / HBM_BYTES_PER_S * 1e3, flops / FP64_FLOPS * 1e3
    b = max(hbm, fp)
    return {"algorithmic_bytes": int(bytes_), "fp64_flops": int(flops), "hbm_bound_ms": round(hbm, 4),
            "fp64_bound_ms": round(fp, 4), "bound": "HBM" if hbm >= fp else "FP64", "bound_ms": round(b, 4),
            "kernel_ms": round(ms, 4), "x_of_bound": round(ms / b, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--variants", type=int, default=1_000_000)
    ap.add_argument("--panel", type=int, default=8192)
    ap.add_argument("--study", default="256,2504")
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("model_bench.py measures on the GPU: no CUDA device")
    n, nv, P = args.samples, args.variants, args.panel
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    report = dict(device_info(), samples=n, variants=nv, panel=P, dtype="int8",
                  peaks={"hbm_bytes_per_s": HBM_BYTES_PER_S, "fp64_flops": FP64_FLOPS}, loadings=[], scoring=[])
    checks = {}
    # ---- fit the panel
    fit = native.NativePca(n, stream=stream.cuda_stream, max_multiplicity=1, num_pc=16)
    buf = torch.zeros(fit.panelBytes(nv, P), dtype=torch.uint8, device="cuda")
    fit.synthPanelsDevice(SEED, 0, nv, 0, buf.data_ptr(), P)
    fit.accumulatePanels(buf.data_ptr(), nv, P)
    fit.finalizeGram()
    fit.computePca(16)
    # ---- loadings (both k against the PCs of one computePca(16): k = 2 must be the first two columns of k = 16)
    Ls = {}
    for k in (16, 2):
        Ls[k] = fit.pcaLoadingsPanels(k, buf.data_ptr(), nv, P)
        ms, reps, tot = kernel_ms(lambda: fit.pcaLoadingsPanels(k, buf.data_ptr(), nv, P), ["model_loadings"], args.min_seconds)
        res = {"k": k, "calls": reps, "kernel_total_ms": round(tot, 2),
               **bound(n * nv + nv * (8 * k + 4), 2.0 * k * n * nv, ms)}
        report["loadings"].append(res)
        print(json.dumps(res), flush=True)
    checks["loadings_k2_equal_first_columns_of_k16"] = bool(
        np.array_equal(Ls[2][0].view(np.int64), Ls[16][0][:, :2].view(np.int64)) and np.array_equal(Ls[2][1], Ls[16][1]))
    vecs, evals, _ = fit.computePca(2)                      # the model: the PCs of computePca(2), as a fitting run has
    L2, c2 = fit.pcaLoadingsPanels(2, buf.data_ptr(), nv, P)
    rng = np.random.default_rng(1)
    sample = np.sort(rng.choice(nv, size=64, replace=False))
    cells = buf.view(-1, n, P)[torch.as_tensor(sample // P, device="cuda"), :, torch.as_tensor(sample % P, device="cuda")]
    X = cells.to(torch.float64).cpu().numpy()              # (64, n)
    want = X @ vecs
    checks["loadings_match_fp64_XtU"] = bool(np.all(np.abs(L2[sample] - want) <= 1e-12 * np.abs(L2).max(axis=0)))
    checks["carriers_exact"] = bool(np.array_equal(c2[sample], X.sum(axis=1).astype(np.int32)))
    terms = fit.pcaModelTerms(2)
    model = type("Model", (), dict(loadings=L2, carriers=c2, n_fitted=n, **terms))
    rows_all = np.arange(nv, dtype=np.int32)
    # fitted samples scored as a study land on their fitted coordinates
    mf = 256
    fitted_copy = buf.view(-1, n, P)[:, :mf, :].contiguous().view(-1)
    with native.NativePca(mf, stream=stream.cuda_stream, max_multiplicity=1, model=model) as sc:
        sc.scorePanels(fitted_copy.data_ptr(), nv, P, rows_all)
        yf, _ = sc.scoreProject(2)
    checks["fitted_copies_on_fitted_coordinates_1e-9"] = bool(np.all(np.abs(yf - vecs[:mf]) <= 1e-9))
    report["fitted_copies_max_abs_diff"] = float(np.abs(yf - vecs[:mf]).max())
    fit.close()
    del fitted_copy
    # ---- scoring vs the projecting context at the same M: the panel's rows, then M study rows (another seed)
    for m in [int(x) for x in args.study.split(",")]:
        sc = native.NativePca(m, stream=stream.cuda_stream, max_multiplicity=1, model=model)
        study = torch.zeros(sc.panelBytes(nv, P), dtype=torch.uint8, device="cuda")
        sc.synthPanelsDevice(SEED + 1, 0, nv, 0, study.data_ptr(), P)
        proj = native.NativePca(n, stream=stream.cuda_stream, max_multiplicity=1, n_projected=m,
                                sample_rows=np.arange(n + m, dtype=np.int32))
        pbuf = torch.cat([buf.view(-1, n, P), study.view(-1, m, P)], dim=1).contiguous().view(-1)

        def gram():
            proj.reset()
            proj.accumulatePanels(pbuf.data_ptr(), nv, P)
        for _ in range(3):
            gram()
        stream.synchronize()
        gms = []
        while sum(gms) < 1e3 * args.min_seconds or len(gms) < 5:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            gram()
            b.record()
            b.synchronize()
            gms.append(a.elapsed_time(b))
        proj.finalizeGram()
        pv, _, _ = proj.computePca(2)
        y_proj = proj.projectPca(2)
        pms, _, _ = kernel_ms(lambda: proj.projectPca(2), ["proj_rowmean", "proj_dot", "proj_finish"], 0.2)

        def score():
            sc.reset()
            sc.scorePanels(study.data_ptr(), nv, P, rows_all)
            return sc.scoreProject(2)
        y, matched = score()
        y_again, _ = score()
        ms, reps, tot = kernel_ms(score, ["model_score", "model_fold"], args.min_seconds)
        res = {"m": m, "k": 2, "calls": reps, "kernel_total_ms": round(tot, 2),
               **bound(m * nv + nv * (8 * 2 + 4 + 4), 2.0 * 2 * m * nv, ms),
               "projecting_gram_ms_median": round(float(np.median(gms)), 4), "project_pca_kernels_ms": round(pms, 4),
               "max_abs_diff_vs_project_pca_over_max_abs_y": [float(np.abs(y[:, c] - y_proj[:, c]).max() /
                                                                    np.abs(y_proj[:, c]).max()) for c in range(2)]}
        checks[f"scores_m{m}_match_project_pca"] = bool(all(d <= 1e-9 for d in res["max_abs_diff_vs_project_pca_over_max_abs_y"]))
        checks[f"scores_m{m}_repeat_bit_identical"] = bool(np.array_equal(y.view(np.int64), y_again.view(np.int64)))
        checks[f"scores_m{m}_all_variants_matched"] = matched == nv
        checks[f"pcs_m{m}_equal_fit"] = bool(np.array_equal(pv, vecs))
        report["scoring"].append(res)
        print(json.dumps(res), flush=True)
        sc.close()
        proj.close()
        del pbuf, study
        torch.cuda.empty_cache()
    report["checks"] = checks
    report["all_checks_pass"] = all(checks.values())
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(report, indent=1) + "\n")
    print(json.dumps({"checks": checks, "all_checks_pass": report["all_checks_pass"]}))
    if not report["all_checks_pass"]:
        raise SystemExit(1)


if __name__ == "__main__":
    main()
