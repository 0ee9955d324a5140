#!/usr/bin/env python
"""bench.py -- genotype-cells/s (N x V) into the Gram on B200, the metric BASELINE.json names.

    python bench.py --gpus N --steps K --warmup W              # this repo's CUDA path (one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU algorithm (oracle port)
    python bench.py ... --dump-outputs DIR                     # also write the last timed step's Gram to DIR/gram.npy

Workload (config.workload): BASELINE.json configs[1] -- 2504 samples x 1 M variants, int8 binary carrier encoding,
per GPU (weak scaling: every rank owns `--variants-per-gpu` variants; 8 ranks x 5 M is configs[2]).  Synthetic
Balding-Nichols-like cohort generated on the device (DESIGN.md "Synthetic generator").

A step = one pass of the hot path over the rank's resident genotype matrix:
    zero S -> tcgen05 Gram kernel over all V variants -> [N > 1: one NCCL all-reduce of S] -> symmetrize.
`value`  = N_samples * V_total * steps / time, inputs resident in HBM (X is 2.5 GB per rank, far larger than the
           126 MB L2, so no flush is needed between iterations), CUDA-event timed, max over ranks.
`e2e`    = the same metric through the public API with HOST inputs: pinned RDD[Seq[Int]] rows (CSR) -> H2D ->
           device encode -> Gram -> centering -> eigensolve -> top-2 PCs back on the host, every step.
`roofline` = the Gram kernel alone against the tensor-core peak (int8 peak taken as 2 x the measured bf16 figure of
           MEASURED_PEAKS.json); numerator = SYRK-minimal ops N (N+1) V (SURVEY.md 8d).
`cpu_baseline` = the oracle's restatement of VariantsPca.scala:182-191 timed on this box's host cores on a FIXED
           sample (32 768 variants, one partition matrix per physical core, median of 5; rank 0, N = 1 only).
Extra legs in the same JSON line (BASELINE configs[2] and [4]; the headline fields above stay configs[1]):
`c3`       = 2504 samples x 5 M variants PER GPU (at --gpus 8 this IS configs[2], 2504 x 40 M), int8 and packed e2m1,
           timed back to back for >= 2 s with its own clock samples: the sustained number, against the sustained peak.
`c5_bf16`  = 10 000 samples x 1.25 M variants per GPU in bf16 (configs[4] is this at 8 GPUs; 1/2/4/8 give the sweep).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

N_SAMPLES = 2504
SEED = 20240901
METRIC = "genotype-cells/sec (N x V) into Gram"
UNIT = "cells/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--samples", type=int, default=N_SAMPLES)
    ap.add_argument("--variants-per-gpu", type=int, default=1_000_000)
    ap.add_argument("--dtype", choices=["i8", "bf16", "e2m1"], default="i8")
    ap.add_argument("--no-alt", action="store_true", help="skip the packed-e2m1 comparison leg")
    ap.add_argument("--panel-variants", type=int, default=int(os.environ.get("VPCA_BENCH_PANEL", "8192")),
                    help="resident cohort layout: panels of this many variants (vpca_accumulate_panels); 0 = row-major")
    ap.add_argument("--reduce", choices=["nccl", "fused", "scatter"], default=os.environ.get("VPCA_BENCH_REDUCE", "scatter"),
                    help="N > 1: 'nccl' = one all-reduce after the Gram kernel; 'fused' = the Gram epilogue adds into every "
                         "rank's Gram over NVLink peer memory (vpca_gram_set_peers); 'scatter' = the epilogue adds into the "
                         "Gram of the rank that owns the row band, then every rank pushes its band to the others (vpca_gram_gather)")
    ap.add_argument("--e2e-steps", type=int, default=-1, help="-1: min(steps, 5); 0 disables the e2e leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eig-check", action="store_true")
    ap.add_argument("--cpu-sample-variants", type=int, default=32768, help="fixed sample of the CPU arm (variants per pass)")
    ap.add_argument("--cpu-repeats", type=int, default=5, help="passes of the CPU arm; the median is reported")
    ap.add_argument("--c3-variants-per-gpu", type=int, default=5_000_000, help="0 disables the c3 / sustained leg")
    ap.add_argument("--c3-seconds", type=float, default=2.0, help="back-to-back duration of the sustained leg")
    ap.add_argument("--c5-samples", type=int, default=10_000)
    ap.add_argument("--c5-variants-per-gpu", type=int, default=1_250_000, help="0 disables the c5_bf16 leg")
    ap.add_argument("--no-legs", action="store_true", help="skip the c3 and c5_bf16 legs (quick kernel A/B runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the Gram of the last one to DIR/gram.npy (see dump_gram)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"bf16_tflops": float(d.get("bf16_tflops", 1590.0)),
                "bf16_tflops_sustained": float(d.get("bf16_tflops_sustained", 1400.0)),
                "hbm_gbs": float(d.get("hbm_gbs", 6650.0)), "source": "measured"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


DUMP_BYTES = 64_000_000


def dump_gram(out_dir, S):
    """--dump-outputs: the symmetrized N x N Gram a step hands its caller, as DIR/gram.npy in float64 (exact for every
    int32 count), so that two builds run with the same arguments can be compared entry for entry.  A Gram larger than
    DUMP_BYTES is sampled: whole rows drawn by a generator seeded with SEED (the same rows on every run), their indices
    in DIR/gram_rows.npy."""
    import numpy as np
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    n = S.shape[0]
    rows_file = out / "gram_rows.npy"
    if 8 * S.size > DUMP_BYTES - 4096:                   # 4096: room for the .npy headers
        rows = np.sort(np.random.default_rng(SEED).choice(n, size=(DUMP_BYTES - 4096) // (8 * (n + 1)), replace=False))
        S = S[rows]
        np.save(rows_file, rows.astype(np.float64))
    else:
        rows_file.unlink(missing_ok=True)
    np.save(out / "gram.npy", S.astype(np.float64))


class ClockSampler(threading.Thread):
    """Samples SM clock, power and throttle reasons through NVML (what nvidia-smi reads) while a region runs."""

    def __init__(self, index: int, period_s: float = 0.01):
        super().__init__(daemon=True)
        self.index, self.period = index, period_s
        self.samples, self.reasons = [], set()
        self._halt = threading.Event()
        self.max_mhz = None
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        while not self._halt.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((mhz, pw))
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2.0)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        mhz = sorted(s[0] for s in self.samples)
        return {"sm_mhz": mhz[len(mhz) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(mhz), "power_w_max": max(s[1] for s in self.samples)}


# ------------------------------------------------------------------------------------------- reference arm
def host_threads():
    """All host threads this process may use (torchrun exports OMP_NUM_THREADS=1; the CPU arm must not obey that)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def physical_cores():
    """Physical cores this process may run on: the partition count of the CPU arm (two hyper-threads of one core share
    the L1/L2 their 25 MB partition matrix streams through, so logical threads only add noise)."""
    logical = host_threads()
    try:
        import psutil
        phys = psutil.cpu_count(logical=False) or logical
        total = psutil.cpu_count(logical=True) or logical
        return max(1, min(logical, int(round(logical * phys / max(1, total)))))
    except Exception:
        return logical


def numa_policy():
    try:
        nodes = len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node")])
    except OSError:
        nodes = 1
    return f"default (first touch: every partition matrix is allocated and zeroed by the thread that fills it), {nodes} NUMA node(s)"


def cpu_similarity_sample(n, variants=32768, threads=None, repeats=5):
    """Time the oracle's getSimilarityMatrix restatement on a FIXED sample: `variants` variants of the benchmark cohort,
    one dense int32 N x N per thread = per Spark partition (VariantsPca.scala:185), summed at the end (:190).
    Returns (median cells/s, info).  A fixed sample keeps the fixed cost (allocating and summing `threads` matrices) in
    the same proportion on every box, so two boxes give comparable numbers."""
    from oracle import oracle
    oracle.build()
    threads = threads or physical_cores()
    oracle.c_set_threads(threads)          # also for the sample generator (torchrun exports OMP_NUM_THREADS=1)
    off, idx = oracle.c_synth_calls(SEED, n, 0, variants)
    nv = len(off) - 1
    times, S = [], None
    for _ in range(max(1, repeats) + 1):   # the first pass warms the thread pool and the page tables: dropped
        t0 = time.perf_counter()
        S = oracle.c_similarity(n, off, idx, threads)
        times.append(time.perf_counter() - t0)
    times = sorted(times[1:]) if len(times) > 1 else times
    med = times[len(times) // 2]
    return n * nv / med, {"variants": nv, "seconds": med, "seconds_all": [round(t, 4) for t in times], "threads": threads,
                          "numa": numa_policy(), "checksum": int(S.trace()), "gram": S}


def cpu_blas_sample(n, nv=65_536, threads=None):
    """Context number so that the CPU comparison is not against a strawman (SURVEY.md 8d "strong CPU"): the same Gram
    as one float32 BLAS product X X^T over `nv` variants (exact: every sum stays below 2^24), all host threads."""
    import numpy as np
    from oracle import oracle
    oracle.build()
    threads = threads or host_threads()
    oracle.c_set_threads(threads)
    X = oracle.c_synth_dense(SEED, n, 0, nv, 0).astype(np.float32)
    try:
        from threadpoolctl import threadpool_limits
        ctx = threadpool_limits(limits=threads)
    except Exception:
        import contextlib
        ctx = contextlib.nullcontext()
    with ctx:
        _ = X[:, :1024] @ X[:, :1024].T            # thread-pool warm-up
        t0 = time.perf_counter()
        G = X @ X.T
        dt = time.perf_counter() - t0
    return {"value": n * nv / dt, "unit": UNIT, "cores": threads,
            "sample": f"{nv} variants x {n} samples, numpy float32 X @ X.T ({dt:.2f} s), exact below 2^24",
            "checksum": int(np.trace(G.astype(np.float64)))}


def cpu_eigensolve_sample(S_host, threads=None):
    """Centering + the MLlib recipe (Cov, LAPACK dgesdd through numpy.linalg.svd, first 2 columns of U) on the host:
    oracle.compute_pca = VariantsPca.scala:198-227 restated.  Timed once on the full N x N matrix."""
    from oracle import oracle
    threads = threads or host_threads()
    try:
        from threadpoolctl import threadpool_limits
        ctx = threadpool_limits(limits=threads)
    except Exception:
        import contextlib
        ctx = contextlib.nullcontext()
    with ctx:
        t0 = time.perf_counter()
        U, sv = oracle.compute_pca(S_host, 2)
        dt = time.perf_counter() - t0
    return {"seconds": dt, "cores": threads, "n": int(S_host.shape[0]),
            "what": "oracle.compute_pca: FP64 centering + Cov = C^T C/(m-1) - ... + numpy.linalg.svd (LAPACK dgesdd), "
                    "first 2 columns of U"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle
    oracle.build()
    n = args.samples
    threads = physical_cores()
    vals, info = [], None
    for i in range(args.warmup + args.steps):        # a step = one pass over the fixed sample
        v, info = cpu_similarity_sample(n, args.cpu_sample_variants, threads, repeats=1)
        if i >= args.warmup:
            vals.append(v)
    if args.dump_outputs:
        dump_gram(args.dump_outputs, info["gram"])
    vals.sort()
    value = vals[len(vals) // 2]                      # median over the timed steps
    nv = info["variants"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * n * nv / value, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": f"{n} samples x {args.variants_per_gpu} variants per GPU (BASELINE configs[1]); each "
                               f"step is a fixed sample of {nv} variants of that cohort",
                   "samples": n, "variants_per_gpu": args.variants_per_gpu},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{nv} variants x {n} samples per step (fixed), median of {len(vals)} steps, "
                                   f"oracle/vpca_oracle.c vo_similarity (VariantsPca.scala:182-191 restated; Spark/JVM not "
                                   f"runnable here), OpenMP, {threads} threads = physical cores of {host_threads()} logical; "
                                   f"Gram only", "threads": threads, "numa": info["numa"],
                         "min_max": [vals[0], vals[-1]],
                         "strong_cpu_blas": cpu_blas_sample(n, threads=threads)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ b200 arm
def build_host_calls(torch, cells, n, nv, dev, chunk=50_000):
    """Pinned-host RDD[Seq[Int]] rows (CSR) of the device-resident binary matrix (setup, untimed).
    `cells(c0, c1)` returns the int32 carrier block of variants [c0, c1)."""
    counts = torch.empty(nv, dtype=torch.int64, device=dev)
    for c0 in range(0, nv, chunk):
        c1 = min(nv, c0 + chunk)
        counts[c0:c1] = cells(c0, c1).sum(dim=0)
    off = torch.zeros(nv + 1, dtype=torch.int64, device=dev)
    off[1:] = torch.cumsum(counts, 0)
    nnz = int(off[-1].item())
    off_h = torch.empty(nv + 1, dtype=torch.int64, pin_memory=True)
    off_h.copy_(off)
    idx_h = torch.empty(max(nnz, 1), dtype=torch.int32, pin_memory=True)
    pos = 0
    for c0 in range(0, nv, chunk):
        c1 = min(nv, c0 + chunk)
        nz = torch.nonzero(cells(c0, c1).t().contiguous())        # sorted by variant, then sample
        m = nz.shape[0]
        idx_h[pos:pos + m].copy_(nz[:, 1].to(torch.int32))
        pos += m
        del nz
    assert pos == nnz
    torch.cuda.synchronize()
    return off_h, idx_h, nnz


def bind_to_gpu_numa_node(index: int) -> str:
    """Pins this rank's threads to the CPUs NVML reports as local to its GPU, so that the pinned staging buffers of the
    e2e legs are first-touched on the GPU's own NUMA node (8 ranks copying 4 GB each per step otherwise cross sockets)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        cpus = sorted(os.sched_getaffinity(0))
        return "rank threads bound to the %d CPUs local to GPU %d (NVML ideal affinity: %d..%d)" % (len(cpus), index, cpus[0], cpus[-1])
    except Exception as exc:
        return "default affinity (%s)" % repr(exc)[:80]


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from spark_examples_b200 import native

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_note = bind_to_gpu_numa_node(local_rank)      # before any pinned host allocation: first touch on the GPU's node
    if world > 1:
        # keep stdout to the one JSON line: NCCL's version / debug banner goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    n, vpg = args.samples, args.variants_per_gpu
    dtype = {"i8": native.DTYPE_I8, "bf16": native.DTYPE_BF16, "e2m1": native.DTYPE_E2M1}[args.dtype]
    eb = {"i8": 1, "bf16": 2, "e2m1": 0.5}[args.dtype]
    tdtype = {"i8": torch.int8, "bf16": torch.bfloat16, "e2m1": torch.uint8}[args.dtype]
    dname = {"i8": "int8", "bf16": "bf16", "e2m1": "e2m1 (4-bit packed cells, fp32 tensor accumulation, exact)"}[args.dtype]
    if args.dtype == "e2m1" and args.panel_variants % 256:
        raise SystemExit("--dtype e2m1 needs --panel-variants % 256 == 0")
    ld = ((vpg + 127) // 128) * 128
    peaks = load_peaks()

    # a non-default torch stream: libvpca orders all its work on it (a NULL handle would mean "private stream"),
    # so torch.cuda.Event timing, NCCL collectives and the library's kernels share one queue
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0
    fused = world > 1 and args.reduce in ("fused", "scatter")
    scatter = world > 1 and args.reduce == "scatter"
    S = torch.zeros((n, n), dtype=torch.int32, device=dev)
    nat = native.NativePca(n, device=local_rank, dtype=dtype, stream=stream, d_gram=0 if fused else S.data_ptr(),
                           max_multiplicity=1)
    if fused:
        # every rank takes part in every collective below, whatever fails locally, so that all ranks fall back together
        handle = None
        try:
            handle = nat.exportIpcHandle()
        except Exception as exc:
            print(f"[bench] rank {rank}: cannot export the Gram for peer access ({exc!r})", file=sys.stderr)
        handles = [None] * world
        dist.all_gather_object(handles, handle)
        ok = 0
        if all(h is not None for h in handles):
            try:
                nat.setPeers(handles, rank, mode="owner_rows" if scatter else "replicate")
                ok = 1
            except Exception as exc:
                print(f"[bench] rank {rank}: peer-memory reduce unavailable ({exc!r})", file=sys.stderr)
        flag = torch.tensor([ok], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            if rank == 0:
                print("[bench] falling back to the NCCL all-reduce", file=sys.stderr)
            nat.close()
            fused = scatter = False
            nat = native.NativePca(n, device=local_rank, dtype=dtype, stream=stream, d_gram=S.data_ptr(), max_multiplicity=1)
    P = args.panel_variants
    if P > 0:
        npan = (vpg + P - 1) // P
        X = torch.empty(nat.panelBytes(vpg, P), dtype=torch.uint8, device=dev)
        nat.synthPanelsDevice(SEED, rank * vpg, vpg, 0, X.data_ptr(), P)
        Xv = (X.view(npan, n, P // 2) if args.dtype == "e2m1" else X.view(tdtype).view(npan, n, P))
    else:
        X = torch.empty((n, ld // 2 if args.dtype == "e2m1" else ld), dtype=tdtype, device=dev)
        nat.synthDenseDevice(SEED, rank * vpg, vpg, 0, X.data_ptr(), ld)
    torch.cuda.synchronize()

    def gram_launch(nt, x):
        if P > 0:
            nt.accumulatePanels(x.data_ptr(), vpg, P)
        else:
            nt.accumulateDenseDevice(x.data_ptr(), vpg, ld)

    def step():
        nat.reset()
        if fused:
            nat.peerBarrier()                  # every rank's Gram is zeroed before anyone adds into it
            gram_launch(nat, X)                # epilogue reds go to all ranks' Grams (or the row's owner) over NVLink
            nat.gatherGram()                   # all contributions have landed (+ pull the other ranks' row bands)
        else:
            gram_launch(nat, X)
            if world > 1:
                dist.all_reduce(S)             # reduceByKey(_ + _) (VariantsPca.scala:190) = one NCCL all-reduce
        nat.finalizeGram()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    st0 = nat.stats()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    barrier()
    clocks = sampler.stop()
    st1 = nat.stats()
    if args.dump_outputs and rank == 0:
        dump_gram(args.dump_outputs, nat.getGram())     # now: the kernel-only timing below leaves an unfinalized Gram
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = n * vpg * world * args.steps / (ms * 1e-3)
    launches = st1["kernel_launches"] - st0["kernel_launches"]

    # ---- Gram kernel alone (roofline numerator / denominator) ----
    kt, gt = [], []
    for _ in range(max(5, min(args.steps, 20))):
        nat.reset()
        if fused:
            nat.peerBarrier()                  # same protocol as step(): nobody adds into a Gram that is being zeroed
        a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        a.record()
        gram_launch(nat, X)
        b.record()
        if fused:
            nat.gatherGram()
        c.record()
        c.synchronize()
        kt.append(a.elapsed_time(b))
        gt.append(b.elapsed_time(c))
    kernel_ms = sum(kt) / len(kt)
    fused_close_ms = sum(gt) / len(gt) if fused else None      # closing barrier(s) + gather, incl. waiting for the slowest peer
    ops = float(n) * (n + 1) * vpg                       # SYRK-minimal ops per launch (SURVEY.md 8d)
    achieved_tops = ops / (kernel_ms * 1e-3) / 1e12
    mxf4 = args.dtype == "e2m1" and os.environ.get("VPCA_E2M1_MXF4", "1") != "0"
    peak_mult = 1.0 if args.dtype == "bf16" else (4.0 if mxf4 else 2.0)      # dense nominal: bf16 2.25, int8/fp8 4.5, fp4 9 PF
    peak = peak_mult * peaks["bf16_tflops"]
    # DRAM traffic of one launch is an ncu number (dram__bytes_read.sum + dram__bytes_write.sum of `ncu --set full`); it
    # cannot be measured inside this run.  The last capture is kept in profiles/r2_gram_traffic.json together with the
    # hash of the kernel source it was taken from: a capture of a different kernel version reads as null, never as stale.
    traffic, traffic_src = None, None
    tp = ROOT / "profiles" / "r2_gram_traffic.json"
    if tp.exists():
        try:
            tj = json.loads(tp.read_text())
            src_hash = native.gramSourceFingerprint()     # code only: comments and whitespace do not count
            ent = tj.get(args.dtype, {})
            if ent.get("kernel_code_sha256_16") == src_hash:
                traffic, traffic_src = ent.get("dram_bytes_per_launch"), ent.get("source")
        except Exception:
            traffic = None
    nominal = {1.0: 2250.0, 2.0: 4500.0, 4.0: 9000.0}[peak_mult]
    roofline = {"bound": "tensor", "achieved": achieved_tops, "peak": peak, "unit": "TFLOP/s",
                "frac": achieved_tops / peak, "traffic": traffic, "traffic_source": traffic_src,
                "kernel": "gram_kernel<cta_group=%d>" % st1["gram_cta_group"], "kernel_ms": kernel_ms,
                "ops_per_launch": ops, "ops_definition": "SYRK-minimal N(N+1)V (int8 MAC = 2 ops)",
                "peak_source": "%g x %s bf16 burst TFLOP/s of MEASURED_PEAKS.json (nominal dense ratios: int8/fp8 = 2 x bf16, "
                               "fp4 = 4 x bf16)" % (peak_mult, peaks["source"]),
                "frac_of_nominal": achieved_tops / nominal, "nominal_peak": nominal,
                "peak_note": ("frac > 1: the denominator is cuBLAS bf16 throughput (x%g), which itself reaches ~75 %% of the "
                              "nominal tensor peak on this pool; read frac_of_nominal as the utilisation" % peak_mult)
                             if achieved_tops > peak else None,
                "hbm_gbs_algorithmic": (n * vpg * eb + 4.0 * n * n) / (kernel_ms * 1e-3) / 1e9,
                "hbm_peak_gbs": peaks["hbm_gbs"]}

    # ---- size-independent parity properties + full-size eigenvector check (untimed) ----
    checks = {}
    step()
    torch.cuda.synchronize()
    if fused:
        S.copy_(torch.from_numpy(nat.getGram()))
        Sref = S.clone()                       # the same cohort reduced with NCCL must give the same matrix
        with native.NativePca(n, device=local_rank, dtype=dtype, stream=stream, d_gram=Sref.data_ptr(),
                              max_multiplicity=1) as natr:
            Sref.zero_()
            gram_launch(natr, X)
            dist.all_reduce(Sref)
            natr.finalizeGram()
            torch.cuda.synchronize()
        checks["fused_reduce_equals_nccl_allreduce"] = bool(torch.equal(S, Sref))
    checks["gram_symmetric"] = bool(torch.equal(S, S.t()))
    def cells(c0, c1):
        """binary carrier block of variants [c0, c1) as int32 (n, c1 - c0), whatever the storage dtype / layout"""
        def block(view, lo, hi):                      # columns [lo, hi) of a row-major (n, width) view
            if args.dtype == "e2m1":
                b = view[:, lo // 2:hi // 2]
                out = torch.empty((n, hi - lo), dtype=torch.int32, device=dev)
                out[:, 0::2] = ((b & 0x0F) != 0).to(torch.int32)
                out[:, 1::2] = ((b >> 4) != 0).to(torch.int32)
                return out
            return (view[:, lo:hi].to(torch.float32) > 0).to(torch.int32)
        if P == 0:
            return block(X, c0, c1)
        parts = []
        for pn in range(c0 // P, (c1 - 1) // P + 1):
            lo, hi = max(c0, pn * P) - pn * P, min(c1, (pn + 1) * P) - pn * P
            parts.append(block(Xv[pn], lo, hi))
        return torch.cat(parts, dim=1)

    if world == 1:
        carriers = torch.zeros(n, dtype=torch.int64, device=dev)
        colsum = torch.zeros(vpg, dtype=torch.float64, device=dev)
        for c0 in range(0, vpg, 100_000):
            c1 = min(vpg, c0 + 100_000)
            blk = cells(c0, c1)
            carriers += blk.sum(dim=1)
            colsum[c0:c1] = blk.sum(dim=0).to(torch.float64)
        checks["diag_equals_carrier_counts"] = bool(torch.equal(torch.diagonal(S).to(torch.int64), carriers))
        s1 = torch.zeros(n, dtype=torch.float64, device=dev)
        for c0 in range(0, vpg, 100_000):
            c1 = min(vpg, c0 + 100_000)
            s1 += cells(c0, c1).to(torch.float64) @ colsum[c0:c1]
        checks["S_times_ones_equals_X_Xt1"] = bool(torch.equal(S.sum(dim=1).to(torch.float64), s1))
    if n > 65535:
        raise SystemExit("bench.py times Gram + eigensolve; vpca_compute_pca (like MLlib's RowMatrix) stops at 65535 "
                         "samples -- use tools/large_n_shard.py for the Gram alone at biobank-scale N")
    nat.computePca(2)                      # first call builds the CUDA graphs of the eigensolver's step loops (one-off)
    ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ee0.record()
    vecs, evals, nz = nat.computePca(2)
    ee1.record()
    ee1.synchronize()
    eig_ms = ee0.elapsed_time(ee1)
    _st = nat.stats()
    eig_info = {"method": {1: "direct", 2: "lanczos", 3: "lanczos->direct"}.get(_st["eig_method"], "?"),
                "lanczos_steps": _st["eig_iterations"]}
    if _st["eig_method"] == 2 and eig_ms > 0:
        # SURVEY 8d: the eigensolve is reported as bytes moved per second.  One step of the persistent Lanczos kernel
        # (n <= 16384) streams the int32 Gram once (N^2 x 4 B, resident in both L2 partitions at N = 2504: the centring is
        # applied to the vector, C is never materialised); the deflated re-run adds 8 steps; the row sums read S once more.
        persist = n <= 16384 and os.environ.get("VPCA_LZ_PERSIST", "1") != "0"
        passes = _st["eig_iterations"] + (8 if persist else 16)
        eig_info["matrix_bytes_streamed"] = int(passes * n * n * (4 if persist else 8) + n * n * (4 if persist else 12))
        eig_info["gb_per_s"] = eig_info["matrix_bytes_streamed"] / (eig_ms * 1e-3) / 1e9
        eig_info["form"] = "persistent cooperative kernel, 3 grid barriers per step" if persist else "five kernels per step (CUDA graph)"
    if not args.no_eig_check and rank == 0:
        Sd = S.to(torch.float64)
        rs = Sd.sum(dim=1)
        C = Sd - (rs / n)[:, None] - (rs / n)[None, :] + rs.sum() / n / n
        w, V = torch.linalg.eigh(C)                       # library checker, not the product path
        Vt = V[:, [-1, -2]].cpu().numpy()
        for c in range(2):
            i = int(np.argmax(np.abs(Vt[:, c])))
            if Vt[i, c] < 0:
                Vt[:, c] = -Vt[:, c]
        err = np.max(np.abs(vecs - Vt), axis=0) / np.max(np.abs(Vt), axis=0)
        checks["eigvec_max_rel_err_vs_torch_eigh"] = float(err.max())
        checks["eigval_rel_err_vs_torch_eigh"] = float(np.max(np.abs(evals - w[[-1, -2]].cpu().numpy()) / abs(float(w[-1]))))

    # ---- end to end through the public API with host inputs ----
    e2e = None
    e2e_steps = args.e2e_steps if args.e2e_steps >= 0 else min(args.steps, 5)
    def agree(ok):
        """True when `ok` holds on EVERY rank.  The legs below contain collectives, so a rank that could not stage its
        host inputs (e.g. pinned memory exhausted with 8 ranks on one host) must take all ranks out of the leg with it."""
        if world == 1:
            return bool(ok)
        t = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return int(t.item()) == 1

    staged = False
    if e2e_steps > 0:
        try:
            off_h, idx_h, nnz = build_host_calls(torch, cells, n, vpg, dev)
            S2 = torch.zeros((n, n), dtype=torch.int32, device=dev)
            nat2 = native.NativePca(n, device=local_rank, dtype=dtype, stream=stream, d_gram=S2.data_ptr(),
                                    max_multiplicity=1)
            staged = True
        except Exception as exc:
            e2e = {"error": "staging the host inputs failed: " + repr(exc)[:250]}
        if not agree(staged):
            staged = False
            if e2e is None:
                e2e = {"error": "skipped: another rank could not stage its host inputs"}
    if staged:
        try:
            def e2e_step():
                nat2.reset()
                nat2.accumulateCallsRaw(-1, off_h.data_ptr(), idx_h.data_ptr(), vpg)     # H2D + encode + Gram
                if world > 1:
                    dist.all_reduce(S2)
                nat2.finalizeGram()
                return nat2.computePca(2)                                                # center + eig + D2H of the PCs

            e2e_step()
            barrier()
            s20 = nat2.stats()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            a.record()
            for _ in range(e2e_steps):
                pcs = e2e_step()
            b.record()
            barrier()
            wall = time.perf_counter() - t0
            s21 = nat2.stats()
            ems = max(a.elapsed_time(b), 0.0)
            if world > 1:
                t = torch.tensor([ems], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ems = float(t.item())
            # same pipeline with the 16-bit index wire format (vpca_accumulate_calls_u16): half the PCIe bytes
            u16 = None
            idx16 = None
            if n <= 65536:
                try:
                    idx16 = torch.empty(max(nnz, 1), dtype=torch.uint16, pin_memory=True)
                    idx16.copy_(idx_h.to(torch.uint16))
                except Exception as exc:
                    idx16 = None
                    u16 = {"error": repr(exc)[:200]}
            if n <= 65536 and agree(idx16 is not None):
                s30 = nat2.stats()

                def e2e_step16():
                    nat2.reset()
                    nat2.accumulateCallsRaw(-1, off_h.data_ptr(), idx16.data_ptr(), vpg, idx_bytes=2)
                    if world > 1:
                        dist.all_reduce(S2)
                    nat2.finalizeGram()
                    return nat2.computePca(2)

                e2e_step16()
                barrier()
                s30 = nat2.stats()
                a16, b16 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a16.record()
                for _ in range(e2e_steps):
                    pcs16 = e2e_step16()
                b16.record()
                barrier()
                s31 = nat2.stats()
                ems16 = a16.elapsed_time(b16)
                if world > 1:
                    t = torch.tensor([ems16], dtype=torch.float64, device=dev)
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                    ems16 = float(t.item())
                u16 = {"value": n * vpg * world * e2e_steps / (ems16 * 1e-3), "ms_per_step": ems16 / e2e_steps,
                       "h2d_bytes_per_step": (s31["h2d_bytes"] - s30["h2d_bytes"]) // e2e_steps,
                       "pcs_match": bool(np.allclose(pcs16[0], vecs, atol=1e-9))}
                del idx16
            # same pipeline fed with one bitmap row per variant (vpca_accumulate_bits): N / 8 bytes per variant on the wire
            bitleg = None
            bits_h = None
            stride = (n + 7) // 8
            try:
                bits_h = torch.empty((vpg, stride), dtype=torch.uint8, pin_memory=True)
                wts = (2 ** torch.arange(8, device=dev, dtype=torch.int32))
                for c0 in range(0, vpg, 50_000):
                    c1 = min(vpg, c0 + 50_000)
                    blk = cells(c0, c1).t().contiguous()                      # (w, n)
                    pad = torch.zeros((blk.shape[0], stride * 8), dtype=torch.int32, device=dev)
                    pad[:, :n] = blk
                    bits_h[c0:c1].copy_((pad.view(-1, stride, 8) * wts).sum(dim=2).to(torch.uint8))
                torch.cuda.synchronize()
            except Exception as exc:
                bits_h = None
                bitleg = {"error": repr(exc)[:200]}
            bits_ok = agree(bits_h is not None)
            try:
                if not bits_ok:
                    raise RuntimeError("skipped: a rank could not stage the bitmap rows")

                def e2e_step_bits():
                    nat2.reset()
                    nat2.accumulateBitsRaw(-1, bits_h.data_ptr(), vpg, stride)
                    if world > 1:
                        dist.all_reduce(S2)
                    nat2.finalizeGram()
                    return nat2.computePca(2)

                e2e_step_bits()
                barrier()
                sb0 = nat2.stats()
                ab, bb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ab.record()
                for _ in range(e2e_steps):
                    pcsb = e2e_step_bits()
                bb.record()
                barrier()
                sb1 = nat2.stats()
                emsb = ab.elapsed_time(bb)
                if world > 1:
                    t = torch.tensor([emsb], dtype=torch.float64, device=dev)
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                    emsb = float(t.item())
                bitleg = {"value": n * vpg * world * e2e_steps / (emsb * 1e-3), "ms_per_step": emsb / e2e_steps,
                          "h2d_bytes_per_step": (sb1["h2d_bytes"] - sb0["h2d_bytes"]) // e2e_steps,
                          "pcs_match": bool(np.allclose(pcsb[0], vecs, atol=1e-9))}
                del bits_h
            except Exception as exc:          # never lose the headline line to an auxiliary leg
                if bitleg is None:
                    bitleg = {"error": repr(exc)[:200]}
            e2e = {"value": n * vpg * world * e2e_steps / (ems * 1e-3), "unit": UNIT,
                   "h2d_bytes_per_step": (s21["h2d_bytes"] - s20["h2d_bytes"]) // e2e_steps,
                   "d2h_bytes_per_step": (s21["d2h_bytes"] - s20["d2h_bytes"]) // e2e_steps,
                   "steps": e2e_steps, "ms_per_step": ems / e2e_steps, "wall_ms_per_step": 1e3 * wall / e2e_steps,
                   "includes": "pinned host CSR rows -> H2D -> encode -> Gram -> centering -> eigensolve -> PCs on host",
                   "nnz": nnz, "pcs_match_resident_path": bool(np.allclose(pcs[0], vecs, atol=1e-9)),
                   # per rank: every rank copies its own shard from its own pinned buffers (this rank's figure; the
                   # step time is the max over ranks)
                   "h2d_gbs_per_rank": (s21["h2d_bytes"] - s20["h2d_bytes"]) / e2e_steps / (ems / e2e_steps * 1e-3) / 1e9,
                   "host_numa": numa_note,
                   "with_uint16_indices": u16, "with_bitmap_rows": bitleg}
            nat2.close()
        except Exception as exc:      # an auxiliary leg must never cost the headline line
            e2e = {"error": repr(exc)[:300]}

    # ---- comparison leg: the same cohort stored as packed 4-bit e2m1 cells (exact; half the bytes per cell) ----
    alt = None
    if args.dtype == "i8" and not args.no_alt:
        S4 = torch.zeros((n, n), dtype=torch.int32, device=dev)
        with native.NativePca(n, device=local_rank, dtype=native.DTYPE_E2M1, stream=stream, d_gram=S4.data_ptr(),
                              max_multiplicity=1) as nat4:
            if P > 0:
                X4 = torch.empty(nat4.panelBytes(vpg, P), dtype=torch.uint8, device=dev)
                nat4.synthPanelsDevice(SEED, rank * vpg, vpg, 0, X4.data_ptr(), P)
            else:
                X4 = torch.empty((n, ld // 2), dtype=torch.uint8, device=dev)
                nat4.synthDenseDevice(SEED, rank * vpg, vpg, 0, X4.data_ptr(), ld)
            t4 = []
            for _ in range(max(5, min(args.steps, 20)) + 2):
                nat4.reset()
                a4, b4 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a4.record()
                gram_launch(nat4, X4)
                b4.record()
                b4.synchronize()
                t4.append(a4.elapsed_time(b4))
            t4 = t4[2:]
            ms4 = sum(t4) / len(t4)
            nat4.finalizeGram()
            torch.cuda.synchronize()
            mx = os.environ.get("VPCA_E2M1_MXF4", "1") != "0"
            alt = {"dtype": "e2m1 (4-bit packed cells in HBM, tcgen05 %s, fp32 accumulation flushed to int32; exact)"
                            % ("kind::mxf4 with unit block scales" if mx else "kind::f8f6f4"),
                   "kernel_ms": ms4, "cells_per_s_kernel": n * vpg / (ms4 * 1e-3),
                   "achieved_tflops_syrk": ops / (ms4 * 1e-3) / 1e12,
                   "frac_of_fp4_peak_4x_bf16" if mx else "frac_of_2x_bf16_peak":
                       ops / (ms4 * 1e-3) / 1e12 / ((4.0 if mx else 2.0) * peaks["bf16_tflops"]),
                   "gram_bit_identical_to_int8_path": bool(torch.equal(S4, S)) if world == 1 else None}
        del X4, S4


    # ---- extra legs (BASELINE configs[2] and [4]); same step protocol as the headline, own contexts, own clock samples ----
    def open_context(n_leg, dtype_code):
        """A NativePca for `n_leg` samples wired like the headline context: fused owner-rows reduce over peer memory when it
        is available on every rank, else a caller-owned Gram that NCCL all-reduces.  Collective: every rank calls it."""
        S_leg = torch.zeros((n_leg, n_leg), dtype=torch.int32, device=dev)
        want_fused = world > 1 and args.reduce in ("fused", "scatter") and n_leg >= 64 * world
        nat_leg = native.NativePca(n_leg, device=local_rank, dtype=dtype_code, stream=stream,
                                   d_gram=0 if want_fused else S_leg.data_ptr(), max_multiplicity=1)
        is_fused = False
        if want_fused:
            handle = None
            try:
                handle = nat_leg.exportIpcHandle()
            except Exception as exc:
                print(f"[bench] rank {rank}: leg context: no IPC export ({exc!r})", file=sys.stderr)
            hs = [None] * world
            dist.all_gather_object(hs, handle)
            ok = 0
            if all(h is not None for h in hs):
                try:
                    nat_leg.setPeers(hs, rank, mode="owner_rows" if args.reduce == "scatter" else "replicate")
                    ok = 1
                except Exception as exc:
                    print(f"[bench] rank {rank}: leg context: peer-memory reduce unavailable ({exc!r})", file=sys.stderr)
            if agree(ok == 1):
                is_fused = True
            else:
                nat_leg.close()
                nat_leg = native.NativePca(n_leg, device=local_rank, dtype=dtype_code, stream=stream, d_gram=S_leg.data_ptr(),
                                           max_multiplicity=1)
        return nat_leg, S_leg, is_fused

    def run_leg(label, n_leg, vpg_leg, dtype_name, min_seconds, max_steps=2000):
        """`min_seconds` of back-to-back steps on a resident shard of vpg_leg variants per GPU."""
        dcode = {"i8": native.DTYPE_I8, "bf16": native.DTYPE_BF16, "e2m1": native.DTYPE_E2M1}[dtype_name]
        ebytes = {"i8": 1.0, "bf16": 2.0, "e2m1": 0.5}[dtype_name]
        nat_l, S_l, fused_l = open_context(n_leg, dcode)
        try:
            Xl = torch.empty(nat_l.panelBytes(vpg_leg, P_leg), dtype=torch.uint8, device=dev)
            nat_l.synthPanelsDevice(SEED, rank * vpg_leg, vpg_leg, 0, Xl.data_ptr(), P_leg)
            torch.cuda.synchronize()

            def leg_step():
                nat_l.reset()
                if fused_l:
                    nat_l.peerBarrier()
                    nat_l.accumulatePanels(Xl.data_ptr(), vpg_leg, P_leg)
                    nat_l.gatherGram()
                else:
                    nat_l.accumulatePanels(Xl.data_ptr(), vpg_leg, P_leg)
                    if world > 1:
                        dist.all_reduce(S_l)
                nat_l.finalizeGram()

            for _ in range(3):
                leg_step()
            barrier()
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            p0.record()
            leg_step()
            p1.record()
            barrier()
            est = torch.tensor([max(p0.elapsed_time(p1), 1e-3)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(est, op=dist.ReduceOp.MAX)       # every rank runs the same number of steps
            k = int(min(max_steps, max(3, -(-min_seconds * 1e3 // float(est.item())))))
            smp = ClockSampler(local_rank)
            smp.start()
            q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            q0.record()
            for _ in range(k):
                leg_step()
            q1.record()
            barrier()
            clk = smp.stop()
            ms_l = q0.elapsed_time(q1)
            if world > 1:
                t = torch.tensor([ms_l], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms_l = float(t.item())
            kern_ms = float(nat_l.stats()["last_gram_ms"])
            if fused_l:
                S_l.copy_(torch.from_numpy(nat_l.getGram()))
            torch.cuda.synchronize()
            # size-independent parity: symmetric, and diag(S)_i = number of variants sample i carries (over all ranks)
            npan = (vpg_leg + P_leg - 1) // P_leg
            carriers = torch.zeros(n_leg, dtype=torch.int64, device=dev)
            for pn in range(npan):
                if dtype_name == "e2m1":
                    blk = Xl.view(npan, n_leg, P_leg // 2)[pn]
                    carriers += ((blk & 0x0F) != 0).sum(dim=1) + ((blk >> 4) != 0).sum(dim=1)
                elif dtype_name == "bf16":
                    carriers += (Xl.view(torch.bfloat16).view(npan, n_leg, P_leg)[pn] != 0).sum(dim=1)
                else:
                    carriers += (Xl.view(torch.int8).view(npan, n_leg, P_leg)[pn] != 0).sum(dim=1)
            if world > 1:
                dist.all_reduce(carriers)
            mult = {"i8": 2.0, "bf16": 1.0, "e2m1": 4.0 if os.environ.get("VPCA_E2M1_MXF4", "1") != "0" else 2.0}[dtype_name]
            ops_l = float(n_leg) * (n_leg + 1) * vpg_leg                      # SYRK-minimal, per GPU
            out = {"workload": f"{n_leg} samples x {vpg_leg} variants per GPU ({vpg_leg * world} total), {dtype_name}",
                   "value": n_leg * vpg_leg * world * k / (ms_l * 1e-3), "unit": UNIT, "steps": k, "seconds": ms_l * 1e-3,
                   "ms_per_step": ms_l / k, "gram_kernel_ms_last": kern_ms,
                   "per_gpu_tops_step": ops_l / (ms_l / k * 1e-3) / 1e12,
                   "per_gpu_tops_kernel": ops_l / (kern_ms * 1e-3) / 1e12 if kern_ms > 0 else None,
                   "frac_of_sustained_peak": ops_l / (ms_l / k * 1e-3) / 1e12 / (mult * peaks["bf16_tflops_sustained"]),
                   "frac_of_nominal_peak": ops_l / (ms_l / k * 1e-3) / 1e12 / (mult * 2250.0),
                   "peak_source": "%g x bf16_tflops_sustained (%s) of MEASURED_PEAKS.json; nominal = %g x 2250 TFLOP/s dense"
                                  % (mult, peaks["source"], mult),
                   "hbm_gbs_algorithmic": (n_leg * vpg_leg * ebytes + 4.0 * n_leg * n_leg) / (ms_l / k * 1e-3) / 1e9,
                   "reduce": "fused peer-memory reduce" if fused_l else ("nccl all-reduce" if world > 1 else "none (1 GPU)"),
                   "clocks": clk,
                   "checks": {"gram_symmetric": bool(torch.equal(S_l, S_l.t())),
                              "diag_equals_carrier_counts": bool(torch.equal(torch.diagonal(S_l).to(torch.int64), carriers))}}
            del Xl
            return out, S_l
        finally:
            nat_l.close()

    legs = {}
    P_leg = args.panel_variants if args.panel_variants > 0 else 8192
    if not args.no_legs and n <= 65535:
        if args.c3_variants_per_gpu > 0:
            for dn in ("i8", "e2m1"):
                try:
                    res, S3 = run_leg("c3", n, args.c3_variants_per_gpu, dn, args.c3_seconds if dn == "i8" else 0.5)
                    if dn == "i8":
                        res["is_baseline_config"] = ("configs[2] (2504 x 40 M at 8 GPUs)" if world == 8 and n == N_SAMPLES and
                                                     args.c3_variants_per_gpu == 5_000_000 else "configs[2] per-GPU shard")
                        legs["c3"] = res
                        S3_i8 = S3
                    else:
                        res["gram_bit_identical_to_int8_leg"] = bool(torch.equal(S3, S3_i8)) if "c3" in legs else None
                        legs["c3_e2m1"] = res
                    del S3
                except Exception as exc:                     # an auxiliary leg must never cost the headline line
                    legs["c3" if dn == "i8" else "c3_e2m1"] = {"error": repr(exc)[:300]}
                    if world > 1:
                        break                                # ranks may be out of step after a failed collective leg
            S3_i8 = None
        if args.c5_variants_per_gpu > 0 and "error" not in legs.get("c3", {}) and "error" not in legs.get("c3_e2m1", {}):
            try:
                torch.cuda.empty_cache()
                res, S5 = run_leg("c5_bf16", args.c5_samples, args.c5_variants_per_gpu, "bf16", 0.4, max_steps=50)
                res["is_baseline_config"] = ("configs[4] (10 000 x 10 M at 8 GPUs)" if world == 8 else
                                             f"configs[4] per-GPU shard: point {world} of the 1/2/4/8 sweep")
                legs["c5_bf16"] = res
                del S5
            except Exception as exc:
                legs["c5_bf16"] = {"error": repr(exc)[:300]}
        torch.cuda.empty_cache()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:      # the CPU arm gets every host core again, not only the ones local to the GPU (bind_to_gpu_numa_node)
            os.sched_setaffinity(0, range(os.cpu_count() or 1))
        except (AttributeError, OSError):
            pass
        v, info = cpu_similarity_sample(n, args.cpu_sample_variants, repeats=args.cpu_repeats)
        cpu = {"value": v, "unit": UNIT, "cores": info["threads"], "kind": "port",
               "sample": f"{info['variants']} variants x {n} samples (fixed sample; median {info['seconds']:.2f} s of "
                         f"{len(info['seconds_all'])} passes), oracle/vpca_oracle.c vo_similarity = VariantsPca.scala:182-191 "
                         f"restated, OpenMP, one partition matrix per physical core; Gram only",
               "threads": info["threads"], "numa": info["numa"], "seconds_all": info["seconds_all"]}
        try:
            cpu["strong_cpu_blas"] = cpu_blas_sample(n)
        except Exception as exc:
            cpu["strong_cpu_blas"] = {"error": repr(exc)[:200]}
        try:                                   # a-4 + a-5 on the host: what vpca_compute_pca (eig_ms above) replaces
            cpu["eigensolve"] = cpu_eigensolve_sample(S.cpu().numpy())
        except Exception as exc:
            cpu["eigensolve"] = {"error": repr(exc)[:200]}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": dname, "data": "synthetic",
            "config": {"workload": f"{n} samples x {vpg} variants per GPU ({vpg * world} total), "
                                   f"{dname} binary carrier genotypes, Gram"
                                   + ("" if world == 1 else (" + fused reduce-scatter / all-gather over peer memory" if scatter else
                                                             " + fused peer-memory reduce" if fused else " + NCCL all-reduce"))
                                   + " + symmetrize (BASELINE configs[1] per GPU; the c3 leg is configs[2]'s per-GPU shard)",
                       "samples": n, "variants_per_gpu": vpg, "parallelism": f"variant-sharded x{world}",
                       "hbm_layout": (f"panels of {P} variants x {n} samples (vpca_accumulate_panels)" if P > 0
                                      else "row-major samples x variants"),
                       "reduce": ("fused reduce-scatter: Gram epilogue red.add into the owner of each Gram row band over NVLink peer "
                                  "memory, then every rank pushes its finished band to the others" if scatter else
                                  "fused: Gram epilogue red.add into every rank's Gram over NVLink peer memory" if fused
                                  else ("nccl all-reduce" if world > 1 else "none (1 GPU)")),
                       "l2_policy": f"input ({n * vpg * eb / 1e9:.2f} GB per rank) larger than L2; no flush between iterations"},
            "clocks": clocks, "gpu_launches": int(launches), "roofline": roofline,
            "eig_ms": eig_ms, "eig": eig_info, "checks": checks, "fused_close_ms": fused_close_ms,
        }
        line.update(legs)
        if alt is not None:
            line["packed_e2m1"] = alt
        if e2e is not None:
            line["e2e"] = e2e
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    nat.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
