#!/usr/bin/env python
"""bench.py -- GWAS markers/sec on the BASELINE.json configuration (n=10,000 x p=1,000,000
SNPs, 1 trait; the gwaslmm marker scan) plus GRM FP64 TFLOP/s.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on host cores

One process per GPU (torchrun for N>1).  Markers are sharded by contiguous column block
across ranks (strong scaling: the 1M-marker problem is fixed); the scan needs no
collective.  A "step" is one pass of the marker scan over the rank's shard: the TMA
streaming kernel + the per-marker finalisation (statistic, SE, beta, -log10 p).

Timed with CUDA events on the library's launching stream (returned through the C ABI) and
cross-checked by wall clock between device synchronisations; max over ranks.
The reference is pure Julia and no Julia runtime exists in this image, so the reference arm
and `cpu_baseline` time the oracle's C/OpenMP restatement of the reference's per-marker
algorithm (kind "port").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "genomicbreedingmodels.jl_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

SEED = 42
KIND_DIPLOID = 0


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=10_000)
    ap.add_argument("--p", type=int, default=1_000_000, help="total markers (sharded over the GPUs)")
    ap.add_argument("--model", default="lmm", choices=["ols", "lmm"])
    ap.add_argument("--e2e-markers", type=int, default=100_000, help="markers in the host-resident e2e sample")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--grm-n", type=int, default=5_000)
    ap.add_argument("--grm-p", type=int, default=100_000)
    ap.add_argument("--no-grm", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-packed", action="store_true")
    ap.add_argument("--cpu-markers", type=int, default=0, help="markers in the CPU sample (0: sized for ~10-20 s)")
    ap.add_argument("--no-multitrait", action="store_true", help="skip the 20-trait batch on the resident shard")
    ap.add_argument("--no-transform", action="store_true", help="skip the pairwise transformation screen (SURVEY 8f-4)")
    ap.add_argument("--transform-l", type=int, default=8192, help="loci in the pairwise screen (l^2 regressions)")
    ap.add_argument("--no-pipeline", action="store_true",
                    help="skip the whole sharded gwaslmm (filter + GRM + all-reduce + PC1 + scan + gather) through gbm_sharded_gwas")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE configs[3] / configs[4] sections")
    ap.add_argument("--stream-markers", type=int, default=12_500,
                    help="configs[4]: markers per rank and step in the host-resident sample (n = 20,000: 2 GB per rank)")
    ap.add_argument("--no-whole-api", action="store_true",
                    help="skip gwasols / gwaslmm(genomes, phenomes) -> Fit through the host mirror against the CPU whole function")
    ap.add_argument("--pipeline-detail", action="store_true",
                    help="N=1 only: also the phase-by-phase single-GPU pipeline incl. ingestion from pageable host memory")
    ap.add_argument("--lmm-markers", type=int, default=0,
                    help="also run the GRM-covariance LMM engine (eigen-rotation GEMM + per-marker delta search) "
                         "on this many markers")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the per-marker outputs of the last timed step as DIR/<name>.npy "
                         "(float64, markers with a result only, their 0-based indices in DIR/marker_index.npy; at most "
                         "64 MB in all, a fixed seeded sample of the markers beyond that)")
    return ap.parse_args()


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region: one streaming
    `nvidia-smi -lms 20` process per region (a fresh nvidia-smi call per sample is too slow
    for a ~100 ms region)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.proc = None
        self._t = None
        self.t_start = self.t_stop = None
        self.stamped = []

    def _reader(self):
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.strip().split(",")]
            if len(parts) >= 7:
                self.stamped.append((time.perf_counter(), parts))

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self._t = threading.Thread(target=self._reader, daemon=True)
            self._t.start()
            time.sleep(0.15)  # let the stream start before the timed region
        except Exception:
            self.proc = None
        self.t_start = time.perf_counter()
        return self

    def __exit__(self, *a):
        self.t_stop = time.perf_counter()
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=3)
            except Exception:
                self.proc.kill()
            if self._t is not None:
                self._t.join(timeout=3)
        inside = [p for (t, p) in self.stamped if self.t_start <= t <= self.t_stop + 0.03]
        self.samples = inside if inside else [p for (_, p) in self.stamped[-3:]]

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                mx.append(float(s[1]))
                for nm, v in zip(names, s[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def log(msg: str):
    """progress on stderr (stdout carries the one JSON line)"""
    if int(os.environ.get("RANK", "0")) == 0:
        print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def shard_bounds(p: int, world: int, rank: int):
    return (p * rank) // world, (p * (rank + 1)) // world


DUMP_BYTES = 64_000_000  # --dump-outputs: all files together, .npy headers included


def dump_outputs(out_dir: str, arrays: dict, p: int, j0: int, world: int):
    """Writes per-marker arrays (this rank holds markers j0 .. j0 + len - 1 of p) as out_dir/<name>.npy in float64 and
    global marker order, from rank 0 of the `world` ranks, with the 0-based indices of the markers written as
    marker_index.npy.  Only markers with a result are written: the scan leaves NaN at markers removed by the
    fixed-locus filter and at degenerate ones, and a caller's fit holds no entry for them.  When the arrays of all p
    markers would exceed DUMP_BYTES, a fixed seeded sample of the markers is taken (the same one in every array)."""
    k = len(arrays) + 1  # + marker_index
    if 8 * k * p + 1024 * k <= DUMP_BYTES:
        idx = np.arange(p)
    else:
        m = (DUMP_BYTES - 1024 * k) // (8 * k)
        idx = np.sort(np.random.default_rng(SEED).choice(p, m, replace=False))
    p_loc = len(next(iter(arrays.values())))
    mine = idx[(idx >= j0) & (idx < j0 + p_loc)]
    local = {name: np.asarray(a, dtype=np.float64)[mine - j0] for name, a in arrays.items()}
    local["marker_index"] = mine.astype(np.float64)
    if world > 1:  # contiguous column blocks: rank order is marker order
        import torch.distributed as dist

        parts = [None] * world
        dist.all_gather_object(parts, local)
        local = {name: np.concatenate([q[name] for q in parts]) for name in local}
    if int(os.environ.get("RANK", "0")) != 0:
        return
    has_result = np.logical_and.reduce([np.isfinite(local[name]) for name in arrays])
    os.makedirs(out_dir, exist_ok=True)
    for name, a in local.items():
        np.save(os.path.join(out_dir, name + ".npy"), a[has_result])
    log(f"outputs of the last timed step: {int(has_result.sum())} markers with a result of {local['marker_index'].size} "
        f"{'' if idx.size == p else 'sampled '}of {p} -> {out_dir}")


# --------------------------------------------------------------------------------------
# CPU arm: the oracle's C/OpenMP restatement of the reference's per-marker loop
# --------------------------------------------------------------------------------------
def synth_block_chunked(n: int, markers: int, chunk: int = 512):
    """synth.block in column chunks (its uint64 temporaries are ~10x the output)."""
    from oracle import synth

    A = np.empty((n, markers), dtype=np.float64, order="F")
    for j0 in range(0, markers, chunk):
        j1 = min(markers, j0 + chunk)
        A[:, j0:j1] = synth.block(SEED, n, j0, j1 - j0, KIND_DIPLOID)
    return A


def cpu_inputs(n: int, p: int):
    from oracle import synth

    y = synth.phenotype(SEED, n, p, KIND_DIPLOID)
    ys = (y - y.mean()) / y.std(ddof=1)
    pc = np.random.default_rng(1).normal(size=n)
    pc -= pc.mean()
    pc /= np.linalg.norm(pc)
    return ys, pc


def cpu_sample_rate(n: int, p: int, markers: int, reps: int = 1):
    """markers/s of the reference algorithm (std filter, standardise, hcat, pinv(X'X), statistic;
    /root/reference/src/gwas.jl:112-115, :129, :241-245) on all host cores."""
    from oracle import cbind

    cbind.use_all_cores()
    A = synth_block_chunked(n, markers)
    ys, pc = cpu_inputs(n, p)
    cbind.gwasols_raw(A[:, :64], ys, pc)  # warm-up (thread pool, page faults)
    # reps passes over the sample (it is far larger than the host's L3, so every pass streams from
    # DRAM like the full problem would); the rate is the mean over all passes
    t0 = time.perf_counter()
    for _ in range(reps):
        cbind.gwasols_raw(A, ys, pc)
    total = time.perf_counter() - t0
    return markers * reps / total, total, cbind.num_threads()


def find_julia():
    """A Julia runtime on this box (SURVEY.md 8d): PATH first, then anything the driver may have installed under
    baseline/_ref/.  None in the build image."""
    import shutil

    exe = shutil.which("julia")
    if exe:
        return exe
    for root, _, files in os.walk(os.path.join(ROOT, "baseline", "_ref")):
        if "julia" in files and os.access(os.path.join(root, "julia"), os.X_OK):
            return os.path.join(root, "julia")
    return None


def julia_reference(model: str):
    """The reference's own gwasols / gwaslmm on its own CPU-runnable case (BASELINE configs[0]: n=300, l=10,000)
    through baseline/reference_gwas.jl, when Julia AND the package are there.  Returns a dict or a reason string."""
    exe = find_julia()
    if exe is None:
        return "no `julia` on PATH or under baseline/_ref/"
    try:
        out = subprocess.run([exe, "--threads=auto,1", os.path.join(ROOT, "baseline", "reference_gwas.jl"), "300", "10000",
                              model, "3"], capture_output=True, text=True, timeout=900)
    except Exception as e:  # noqa: BLE001
        return f"julia found at {exe} but the run failed: {e}"
    for ln in out.stdout.splitlines():
        if ln.startswith("reference_gwas "):
            f = ln.split()
            return {"julia": exe, "n": int(f[1]), "l": int(f[2]), "model": f[3], "seconds_per_call": float(f[4]),
                    "threads": int(f[5]), "blas_threads": int(f[6]), "markers_per_s": int(f[2]) / float(f[4])}
    return f"julia found at {exe} but GenomicBreedingModels did not run: {(out.stderr or out.stdout)[-300:]}"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import cbind

    cbind.use_all_cores()
    n = args.n
    # bounded sample: ~1 s of CPU work per step, at most 2 GB of genotypes
    rate0, _, cores = cpu_sample_rate(n, args.p, 512)
    markers = args.cpu_markers or int(max(512, min(25_000, rate0 * 1.0)))
    A = synth_block_chunked(n, markers)
    ys, pc = cpu_inputs(n, args.p)
    for _ in range(args.warmup):
        cbind.gwasols_raw(A[:, : min(markers, 2048)], ys, pc)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        stat_ols, stat_lmm, _ = cbind.gwasols_raw(A, ys, pc)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"stat_ols": stat_ols, "stat_lmm": stat_lmm}, markers, 0, 1)
    value = markers * args.steps / dt
    sample = f"{markers} of {args.p} markers per step (n={n}), C/OpenMP restatement of gwas.jl:112-115,:129,:241-245"
    line = {
        "impl": "reference", "metric": "GWAS markers/sec", "value": value, "unit": "markers/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"gwas{args.model} marker scan n={n} p={args.p} 1 trait (BASELINE configs[2])",
                   "sample": sample},
        "cpu_baseline": {"value": value, "unit": "markers/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "markers/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference is pure Julia; no Julia runtime in the image: oracle port timed (DESIGN.md)",
    }
    jr = julia_reference(args.model)
    line["julia_reference"] = jr  # the reference itself on BASELINE configs[0] when a runtime exists, else why not
    if isinstance(jr, dict):
        line["note"] = ("a Julia runtime was found: julia_reference holds the UNMODIFIED reference's own time on its "
                        "CPU-runnable case (configs[0]); value stays the port on the configs[2] sample for comparability")
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------------------
def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    # NCCL / libraries may print banners on stdout; keep stdout for the one JSON line
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist

    import gbm_b200
    from gbm_b200 import _lib
    from oracle import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    gbm_b200.init(local_rank)
    lib = _lib.load()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n, p = args.n, args.p
    j0, j1 = shard_bounds(p, world, rank)
    p_loc = j1 - j0
    model = _lib.MODEL_LMM if args.model == "lmm" else _lib.MODEL_OLS

    # ---- inputs, resident in HBM before the timed region -------------------------------
    dm = gbm_b200.DeviceMatrix.generate(SEED, n, p_loc, KIND_DIPLOID, col0=j0)
    y = synth.phenotype(SEED, n, p, KIND_DIPLOID)
    ys = (y - y.mean()) / y.std(ddof=1)
    pc = np.random.default_rng(1).normal(size=n)  # stand-in covariate for the scan-only step
    pc -= pc.mean()
    pc /= np.linalg.norm(pc)
    Y = np.asfortranarray(ys[:, None])
    C = np.asfortranarray(pc[:, None])
    # outputs stay on the device (l x 4 doubles + filter mask)
    outs = {k: torch.empty(p_loc, dtype=torch.float64, device="cuda") for k in ("beta", "se", "stat", "nlp", "mean", "sd")}
    keep = torch.empty(p_loc, dtype=torch.uint8, device="cuda")

    plan = gbm_b200.ScanPlan(dm, Y, C, model=model)  # y / PC1 prepared and resident before the timed region

    def step():
        # one pass over the shard: streaming-sums kernel + finalisation kernel, device outputs in place
        return plan.run(outs["beta"], outs["se"], outs["stat"], outs["nlp"], outs["mean"], outs["sd"], keep)

    log(f"scan step: {p_loc} markers on this rank")
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    main_ms, kern_ms = [], []
    with ClockSampler(local_rank) as clocks:
        t0 = time.perf_counter()
        for _ in range(args.steps):
            tm = step()  # returns after a stream synchronise
            main_ms.append(tm["main_ms"])
            kern_ms.append(tm["kernel_ms"])
        barrier()
        wall = time.perf_counter() - t0
    dev_s = sum(kern_ms) * 1e-3  # CUDA-event time of all kernels of the K steps on this rank
    t = torch.tensor([dev_s, wall, float(np.mean(main_ms))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_s, wall, main_avg_ms = (float(x) for x in t.cpu())
    value = p * args.steps / dev_s
    wall_value = p * args.steps / wall
    if args.dump_outputs:  # before the packed-copy section below reuses the output buffers
        dump_outputs(args.dump_outputs, {"beta": outs["beta"].cpu(), "se": outs["se"].cpu(), "stat": outs["stat"].cpu(),
                                         "neglog10p": outs["nlp"].cpu(), "mean": outs["mean"].cpu(),
                                         "sd": outs["sd"].cpu()}, p, j0, world)

    peak, peak_src = measured_peaks()
    algo_bytes = 8.0 * n * p_loc  # SURVEY 8d: 8n bytes per marker, each genotype read once
    achieved = algo_bytes / (main_avg_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "scan_traffic.json")
    if os.path.exists(tpath):  # dram__bytes_read+write of this kernel from the committed ncu --set full capture
        with open(tpath) as f:
            tj = json.load(f)
        if tj.get("n") == n:
            traffic = tj["dram_bytes_per_marker"] * p_loc
    roofline = {"bound": "hbm", "kernel": "scan_sums_kernel<16,2>", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": algo_bytes, "avg_launch_ms": main_avg_ms,
                "note": "peak is MEASURED_PEAKS.json's copy bandwidth (a copy's read + write bytes); this kernel only "
                        "reads, and a read-only stream runs above that figure -- ncu: dram__bytes_read = 1.0008 x the "
                        "algorithmic bytes (profiles/r01_ncu_full_scan_final.md)"}
    keep_count = int(keep.sum().item())

    line = {
        "metric": "GWAS markers/sec", "value": value, "unit": "markers/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": dev_s / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"gwas{args.model} marker scan n={n} p={p} 1 trait, PC1 covariate (BASELINE configs[2])",
                   "n": n, "p": p, "markers_per_gpu": p_loc, "sharding": f"column-block x{world}",
                   "cache": "inputs larger than L2 (shard >= 10 GB vs 126 MB L2)", "markers_kept": keep_count,
                   "generator": "oracle/synth.py diploid, on-device"},
        "wall_value": wall_value, "roofline": roofline, "gpu_launches": 2 * args.steps,
    }

    # ---- rank-0 extras: clocks, e2e, GRM, CPU baseline ---------------------------------
    line["clocks"] = clocks.summary()

    # ---- compact storage (1 byte per genotype; SURVEY 8f-3): same step on the packed copy ----
    if not args.no_packed:
        pk = dm.pack()
        if pk is not None:
            pplan = gbm_b200.ScanPlan(pk, Y, C, model=model)
            for _ in range(3):
                pplan.run(outs["beta"], outs["se"], outs["stat"], outs["nlp"], outs["mean"], outs["sd"], keep)
            barrier()
            pk_ms, pm_ms = [], []
            for _ in range(args.steps):
                tm = pplan.run(outs["beta"], outs["se"], outs["stat"], outs["nlp"], outs["mean"], outs["sd"], keep)
                pk_ms.append(tm["kernel_ms"])
                pm_ms.append(tm["main_ms"])
            barrier()
            tt = torch.tensor([sum(pk_ms) * 1e-3, float(np.mean(pm_ms))], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            pdev_s, pmain = (float(x) for x in tt.cpu())
            pach = 1.0 * n * p_loc / (pmain * 1e-3) / 1e9
            line["packed"] = {"metric": "GWAS markers/sec, 1-byte dosage codes resident in HBM",
                              "value": p * args.steps / pdev_s, "unit": "markers/s",
                              "roofline": {"bound": "hbm", "kernel": "scan_sums_u8_tc_kernel (tcgen05 kind::i8 dots)", "achieved": pach,
                                           "peak": peak, "unit": "GB/s", "frac": pach / peak,
                                           "algorithmic_bytes_per_launch": 1.0 * n * p_loc, "avg_launch_ms": pmain},
                              "note": "not the graded Float64 path: algorithmic bytes are n per marker here"}
            pplan.free()
            pk.free()

    # ---- multi-trait batch (BASELINE configs[4] shape: 20 traits, one covariate) on the resident shard:
    #      21 side vectors in one pass on the FP64 tensor pipe (csrc/scan_mt.cu) ----
    if rank == 0 and not args.no_multitrait:
        T = 20
        Ymt = np.asfortranarray(np.random.default_rng(7).normal(size=(n, T)))
        mplan = gbm_b200.ScanPlan(dm, Ymt, C, model=_lib.MODEL_OLS)
        mstat = torch.empty(p_loc * T, dtype=torch.float64, device="cuda")
        for _ in range(2):
            mplan.run(stat=mstat)
        mk, mm = [], []
        for _ in range(3):
            tm = mplan.run(stat=mstat)
            mk.append(tm["kernel_ms"])
            mm.append(tm["main_ms"])
        mplan.free()
        del mstat
        ms, main = float(np.median(mk)), float(np.median(mm))
        nt = (T + 1 + 1 + 7) // 8  # [1 | PC1 | 20 traits] in 8-column MMA blocks
        line["multi_trait"] = {
            "workload": f"gwasols batch of {T} traits + 1 covariate on this rank's {p_loc} markers (n={n})",
            "kernel_ms": ms, "sums_kernel_ms": main, "marker_trait_tests_per_s": p_loc * T / (ms * 1e-3),
            "markers_per_s": p_loc / (ms * 1e-3), "hbm_GBps": 8.0 * n * p_loc / (main * 1e-3) / 1e9,
            "dmma_tflops": 2.0 * n * p_loc * 8 * nt / (main * 1e-3) / 1e12,
            "note": "one pass over the genotypes; FP64 tensor pipe (DMMA m8n8k4) for the 22 dots per marker"}

    if not args.no_e2e:
        log("e2e from host memory")
        line.update(run_e2e(args, gbm_b200, _lib, lib, n, p_loc, j0, world, model, Y, C, barrier))

    plan.free()
    # ---- the whole sharded gwaslmm (north_star's target run), every rank takes part: ONE collective call into the
    #      library (gbm_sharded_gwas), NCCL inside it ----
    grp = None
    if not (args.no_pipeline and args.no_configs):
        from gbm_b200 import multigpu

        grp = (multigpu.Group.from_torch_distributed() if world > 1
               else multigpu.Group.from_rank(multigpu.Group.unique_id(), 1, 0))
    if not args.no_pipeline:
        log("whole sharded gwaslmm")
        res = run_pipeline_group(gbm_b200, _lib, grp, dm, n, p, ys, world, rank)
        if rank == 0:
            line["pipeline"] = res
        dm = None
    if dm is not None:
        dm.free()
    if not args.no_configs:
        # BASELINE configs[3]: grmploidyaware + gwaslmm on tetraploid frequencies, n = 2,000 x p = 500,000
        log("configs[3] tetraploid")
        res = run_config3_tetraploid(gbm_b200, _lib, grp, world, rank, measured_peaks()[0])
        if rank == 0:
            line["config3_tetraploid"] = res
        # BASELINE configs[4]: 20 traits x n = 20,000 x p = 2,000,000 streamed from host memory
        log("configs[4] multi-trait stream")
        res = run_config4_stream(args, gbm_b200, _lib, lib, world, rank, j0, barrier)
        if rank == 0:
            line["config4_multitrait_stream"] = res
    if grp is not None:
        grp.free()

    if rank == 0 and not args.no_grm:
        log("GRM")
        gn, gp = args.grm_n, args.grm_p
        gm = gbm_b200.DeviceMatrix.generate(SEED, gn, gp, KIND_DIPLOID)
        dK = torch.empty(gn * gn, dtype=torch.float64, device="cuda")
        tfs = []
        for i in range(4):
            _, tf = gm.grm(_lib.GRM_SIMPLE, 2, 0, out=dK)
            if i:
                tfs.append(tf)
        # the same GRM from the packed (1-byte dosage) copy: exact integer contraction on the
        # tcgen05 INT8 tensor cores (csrc/grm_i8.cu)
        i8 = None
        gk = gm.pack()
        if gk is not None:
            tfi = []
            for i in range(4):
                _, tf = gk.grm(_lib.GRM_SIMPLE, 2, 0, out=dK)
                if i:
                    tfi.append(tf)
            gk.free()
            tf8 = float(np.median(tfi))
            i8 = {"metric": "GRM from 1-byte dosage codes, tcgen05 kind::i8 (exact)", "value": tf8,
                  "unit": "TFLOP/s-equivalent, n(n+1)p / time (incl. centring passes)",
                  "ms": gn * (gn + 1) * gp / tf8 / 1e9, "speedup_vs_fp64_dmma": tf8 / float(np.median(tfs))}
        gm.free()
        # cuBLAS DGEMM peak on this box (the practical FP64 tensor roofline)
        a = torch.randn(8192, 8192, dtype=torch.float64, device="cuda")
        b = torch.randn(8192, 8192, dtype=torch.float64, device="cuda")
        torch.matmul(a, b)
        best = 0.0
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            torch.cuda.synchronize()
            best = max(best, 2 * 8192 ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        # ... and SUSTAINED: back to back for ~1.5 s (the figure a long GEMM-bound phase such as the GRM sees)
        reps = max(4, int(1.5 * best * 1e12 / (2 * 8192 ** 3)))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        sustained = reps * 2 * 8192 ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12
        del a, b, dK
        line["grm"] = {"metric": "GRM FP64 TFLOP/s", "value": float(np.median(tfs)), "unit": "TFLOP/s",
                       "flops_convention": "n(n+1)p (SYRK)", "n": gn, "p": gp,
                       "workload": f"grmsimple n={gn} p={gp} diploid (BASELINE configs[1])",
                       "cublas_dgemm_8192_tflops": best, "frac_of_cublas_dgemm": float(np.median(tfs)) / best,
                       "cublas_dgemm_8192_tflops_sustained": sustained,
                       "frac_of_cublas_dgemm_sustained": float(np.median(tfs)) / sustained,
                       "datasheet_fp64_tflops": 40.0, "frac_of_datasheet": float(np.median(tfs)) / 40.0,
                       "roofline": {"bound": "tensor", "kernel": "grm_dmma_kernel", "achieved": float(np.median(tfs)),
                                    "peak": sustained, "unit": "TFLOP/s", "frac": float(np.median(tfs)) / sustained,
                                    "peak_source": "cuBLAS DGEMM 8192^3 back to back for ~1.5 s in this run "
                                                   "(MEASURED_PEAKS.json has no FP64 figure); burst = cublas_dgemm_8192_tflops",
                                    "traffic": None}}
        if i8 is not None:
            line["grm_int8"] = i8

    if rank == 0 and not args.no_transform:
        line["transform2"] = run_transform2(gbm_b200, n, args.transform_l)

    if rank == 0 and world == 1 and not args.no_whole_api:
        line["whole_api"] = run_whole_api(gbm_b200, with_cpu=not args.no_cpu)

    if rank == 0 and world == 1 and args.pipeline_detail:
        line["pipeline_detail"] = run_pipeline(gbm_b200, _lib, n, p_loc, j0, ys)

    if rank == 0 and args.lmm_markers > 0:
        line["lmm_rotation_engine"] = run_lmm(gbm_b200, _lib, n, args.lmm_markers)

    if rank == 0 and world == 1 and not args.no_cpu:  # reported at N=1 only
        rate0, _, cores = cpu_sample_rate(n, p, 512)
        markers = args.cpu_markers or int(max(1024, min(40_000, rate0 * 12.0)))  # <= 3.2 GB of genotypes
        reps = int(max(1, min(400, round(rate0 * 12.0 / markers))))  # ~12 s of CPU work in all
        rate, secs, cores = cpu_sample_rate(n, p, markers, reps)
        line["cpu_baseline"] = {"value": rate, "unit": "markers/s", "cores": cores, "kind": "port",
                                "sample": f"{reps} passes over {markers} of {p} markers (n={n}) in {secs:.1f} s; C/OpenMP restatement of "
                                          "the reference's per-marker loop (gwas.jl:112-115,:129,:241-245); the "
                                          "reference is Julia and cannot run in this image"}

    sys.stdout.flush()
    os.dup2(real_stdout, 1)
    if rank == 0:
        print(json.dumps(line), flush=True)
    os.dup2(2, 1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def run_pipeline(gbm_b200, _lib, n, p_loc, j0, ys):
    """Whole gwaslmm once on one GPU: colstats/filter + GRM (DMMA) + K standardise + PC1
    (cuSOLVER) + scan.  The eigen step is timed separately, as BASELINE.json asks."""
    import torch

    out = {}
    # one-off library initialisation (cuSOLVER/cuBLAS handles, kernel images) on a toy problem
    wm = gbm_b200.DeviceMatrix.generate(SEED, 256, 512, KIND_DIPLOID)
    wK, _ = wm.grm(_lib.GRM_SIMPLE, 2, 0)
    gbm_b200.kstd_pc1(wK, want_kstd=False)
    wm.free()
    dm = gbm_b200.DeviceMatrix.generate(SEED, n, p_loc, KIND_DIPLOID, col0=j0)
    dK = torch.empty(n * n, dtype=torch.float64, device="cuda")
    for attempt in ("cold", "warm"):  # the first pass pays cuSOLVER's lazy initialisation for this size
        t_all = time.perf_counter()
        t0 = time.perf_counter()
        st = dm.colstats()
        out["colstats_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        _, tf = dm.grm(_lib.GRM_SIMPLE, 2, 0, out=dK)
        out["grm_s"] = time.perf_counter() - t0
        out["grm_tflops"] = tf
        t0 = time.perf_counter()
        pc, eig_ms = gbm_b200.kstd_pc1_device(dK.data_ptr(), n)
        out["kstd_pc1_s"] = time.perf_counter() - t0
        out["eig_s"] = eig_ms * 1e-3
        t0 = time.perf_counter()
        res = dm.scan(ys, pc[:, None], model=_lib.MODEL_LMM)
        out["scan_s"] = time.perf_counter() - t0
        out["scan_kernel_ms"] = _lib.last_timing()["main_ms"]
        out["scan_timing"] = _lib.last_timing()
        if attempt == "cold":
            out["first_pass_total_s"] = time.perf_counter() - t_all
    out["markers_kept"] = int(st["idx_cols"].size)
    out["max_neglog10p"] = float(np.nanmax(res["neglog10p"]))
    tot = out["colstats_s"] + out["grm_s"] + out["kstd_pc1_s"] + out["scan_s"]
    out["total_s"] = tot
    out["markers_per_s_whole_gwaslmm"] = p_loc / tot
    # the same pipeline on the packed (1-byte dosage) copy: u8 scan kernels + exact INT8 tensor-core GRM
    t0 = time.perf_counter()
    pk = dm.pack()
    pack_s = time.perf_counter() - t0
    if pk is not None:
        pkd = {"pack_s": pack_s}
        for attempt in ("cold", "warm"):
            t0 = time.perf_counter()
            st2 = pk.colstats()
            pkd["colstats_s"] = time.perf_counter() - t0
            t0 = time.perf_counter()
            _, tf = pk.grm(_lib.GRM_SIMPLE, 2, 0, out=dK)
            pkd["grm_s"] = time.perf_counter() - t0
            pkd["grm_tflops_equivalent"] = tf
            t0 = time.perf_counter()
            pc2, eig_ms = gbm_b200.kstd_pc1_device(dK.data_ptr(), n)
            pkd["kstd_pc1_s"] = time.perf_counter() - t0
            pkd["eig_s"] = eig_ms * 1e-3
            t0 = time.perf_counter()
            res2 = pk.scan(ys, pc2[:, None], model=_lib.MODEL_LMM)
            pkd["scan_s"] = time.perf_counter() - t0
        tot2 = pkd["colstats_s"] + pkd["grm_s"] + pkd["kstd_pc1_s"] + pkd["scan_s"]
        pkd["total_s"] = tot2
        pkd["markers_per_s_whole_gwaslmm"] = p_loc / tot2
        keep = res["keep"]
        d = np.abs(res2["stat"][keep, 0] - res["stat"][keep, 0])
        pkd["max_abs_diff_z_vs_float64_pipeline"] = float(np.nanmax(d))
        pkd["filter_identical"] = bool(np.array_equal(st2["idx_cols"], st["idx_cols"]))
        out["packed_int8"] = pkd
        pk.free()
    # the same from HOST memory (what the drop-in API gets: a pageable Float64 matrix): ingestion by
    # gbm_matrix_upload_compact (host cores pack on the way) + the packed pipeline above
    fh = {}
    try:
        host = np.empty((p_loc, n))  # C-order (p, n) == n x p column-major; pageable, like a Julia Array
        dm.download_into(host)
        dm.free()
        dm = None
        A = host.T  # F-contiguous view n x p
        for attempt in ("cold", "warm"):
            t_all = time.perf_counter()
            m = gbm_b200.DeviceMatrix.upload_compact(A)
            fh["upload_s"] = time.perf_counter() - t_all
            fh["packed"] = bool(m.packed)
            st3 = m.colstats()
            _, tf = m.grm(_lib.GRM_SIMPLE, 2, 0, out=dK)
            pc3, eig_ms = gbm_b200.kstd_pc1_device(dK.data_ptr(), n)
            res3 = m.scan(ys, pc3[:, None], model=_lib.MODEL_LMM)
            fh["total_s"] = time.perf_counter() - t_all
            m.free()
        fh["markers_per_s_whole_gwaslmm_from_host"] = p_loc / fh["total_s"]
        fh["upload_GBps_f64_equiv"] = 8.0 * n * p_loc / fh["upload_s"] / 1e9
        fh["max_neglog10p"] = float(np.nanmax(res3["neglog10p"]))
        del host, A
    except MemoryError as e:
        fh["skipped"] = f"host matrix does not fit: {e}"
    out["from_host"] = fh
    if dm is not None:
        dm.free()
    return out


def run_e2e(args, gbm_b200, _lib, lib, n, p_loc, j0, world, model, Y, C, barrier):
    """The metric end to end through the C-ABI call a host makes with HOST buffers: gbm_scan_host(A, ...) -> results,
    host -> device copies inside the timed region.  The headline `e2e` is timed from PAGEABLE memory -- what a Julia
    `Array` (genomes.allele_frequencies) is -- through the API's default path (blocks that are all dosage codes
    are packed to 1 byte per genotype by the host cores before crossing PCIe; the data here is diploid dosages).
    Also reported: the same from pinned memory, and plain Float64 copies (GBM_SCAN_HOST_NO_PACK: what continuous
    allele frequencies get) from pageable and from pinned memory, next to the link's plain-copy rate."""
    import ctypes

    import torch
    import torch.distributed as dist

    pe = min(args.e2e_markers, p_loc)
    pinned = torch.empty((pe, n), dtype=torch.float64, pin_memory=True)  # (p, n) C-order == n x p column-major
    sub = gbm_b200.DeviceMatrix.generate(SEED, n, pe, KIND_DIPLOID, col0=j0)
    info = sub.info()
    assert info["lda"] == n
    cudart = ctypes.CDLL("libcudart.so.12")
    rc = cudart.cudaMemcpy(ctypes.c_void_p(pinned.data_ptr()), ctypes.c_void_p(info["device_ptr"]),
                           ctypes.c_size_t(8 * n * pe), ctypes.c_int(2))  # device -> host, untimed set-up
    assert rc == 0, rc
    sub.free()
    pageable = np.empty((pe, n))  # plain malloc'ed memory, like a Julia Array
    pageable[:] = pinned.numpy()
    hout = {k: np.zeros(pe) for k in ("beta", "se", "stat", "nlp", "mean", "sd")}
    hkeep = np.zeros(pe, dtype=np.uint8)

    def step(buf, flags):
        _lib.check(lib.gbm_scan_host(_lib.ptr(buf), n, pe, n, _lib.ptr(Y), 1, n, _lib.ptr(C), 1, n, model, flags,
                                     _lib.ptr(hout["beta"]), _lib.ptr(hout["se"]), _lib.ptr(hout["stat"]),
                                     _lib.ptr(hout["nlp"]), _lib.ptr(hout["mean"]), _lib.ptr(hout["sd"]), _lib.ptr(hkeep)))

    def timed(buf, flags):
        step(buf, flags)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            step(buf, flags)
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        ltm = _lib.last_timing()
        return {"value": pe * world * args.e2e_steps / dt, "unit": "markers/s",
                "h2d_bytes_per_step": ltm["h2d_bytes"] + 16 * n, "d2h_bytes_per_step": pe * (6 * 8 + 1),
                "host_read_gbps": 8.0 * n * pe * world * args.e2e_steps / dt / 1e9,
                "blocks_as_codes": ltm["packed_blocks"], "blocks_packed_by_host": ltm["host_packed_blocks"]}

    # the link itself: plain pinned H2D copy of the same buffer (reference point)
    dev = torch.empty((pe, n), dtype=torch.float64, device="cuda")
    dev.copy_(pinned, non_blocking=True)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    dev.copy_(pinned, non_blocking=True)
    ev1.record()
    torch.cuda.synchronize()
    h2d_peak = 8.0 * n * pe / (ev0.elapsed_time(ev1) * 1e-3) / 1e9
    del dev
    sample = f"{pe} host-resident markers per GPU per step through gbm_scan_host (n={n})"
    out = {}
    e = timed(pageable, 0)
    e.update(sample=sample, host_memory="pageable (malloc), as a Julia Array", host_threads=len(os.sched_getaffinity(0)),
             note="API default: column blocks handed out dynamically to the host cores (pack to 1-byte codes, exactness-"
                  "checked, then H2D) and/or the copy engine (Float64 H2D, packed on the device)")
    out["e2e"] = e
    if not args.no_packed:
        e = timed(pinned, 0)
        e.update(sample=sample, host_memory="pinned")
        out["e2e_pinned"] = e
    for name, buf in (("e2e_float64_copies", pageable), ("e2e_float64_copies_pinned", pinned)):
        e = timed(buf, _lib.SCAN_HOST_NO_PACK)
        e.update(sample=sample, host_memory="pageable" if buf is pageable else "pinned",
                 h2d_gbps_per_gpu=e["host_read_gbps"] / world, h2d_link_gbps_plain_copy=h2d_peak,
                 frac_of_link=e["host_read_gbps"] / world / h2d_peak,
                 bound="PCIe host->device link: 8n bytes per marker must cross it",
                 note="gbm_scan_host with GBM_SCAN_HOST_NO_PACK: what continuous (non-dosage) allele frequencies get")
        out[name] = e
    return out


def run_pipeline_group(gbm_b200, _lib, grp, dm, n, p, ys, world, rank):
    """Whole gwaslmm (/root/reference/src/gwas.jl:329-399 after extractxyetc) on all ranks through the library's
    group API: gbm_group_create_rank + gbm_sharded_adopt + gbm_sharded_gwas.  Each rank holds its column block;
    filter local, GRM partials summed with ONE NCCL all-reduce, K standardisation + PC1 with the columns of K
    sharded (one n-vector all-reduce per Lanczos step), scan local, results gathered in locus order on every
    rank.  Both storages: Float64 slabs (FP64 DMMA GRM) and 1-byte dosage codes (u8 scan, tcgen05 INT8 GRM).
    Times are the library's host wall clock per phase, max over ranks; the second (warm) call is reported.
    Consumes dm."""
    import torch
    import torch.distributed as dist

    from gbm_b200 import multigpu

    out = {"world": world, "n": n, "p": p, "api": "gbm_sharded_gwas (one collective call; NCCL inside libgbm_b200.so)"}
    keys = ("colstats_ms", "grm_ms", "allreduce_ms", "kstd_pc1_ms", "eig_ms", "scan_ms", "gather_ms", "total_ms",
            "scan_kernel_ms")
    m = dm
    for storage in ("float64", "packed"):
        if storage == "packed":
            t0 = time.perf_counter()
            m = dm.pack()
            pack_s = time.perf_counter() - t0
            dm.free()
            ok = torch.tensor([0.0 if m is None else 1.0], device="cuda")
            if world > 1:
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if ok.item() < 0.5:
                break
        sm = multigpu.ShardedMatrix.adopt(grp, [m])
        res = None
        for attempt in ("cold", "warm"):
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            # Fit needs b_hat = the statistic (gwas.jl:245, :385); -log10 p is what `verbose` plots (:252, :392).
            # The output arrays of the first call are reused by the second (like a preallocated Fit.b_hat).
            res = sm.gwas(ys, model=_lib.MODEL_LMM, grm_type=_lib.GRM_SIMPLE, want=("stat", "neglog10p"), out=res)
            wall = time.perf_counter() - t0
            if attempt == "cold":
                cold_total = res["timing"]["total_ms"]
        tm = res["timing"]
        tt = torch.tensor([tm[k] for k in keys] + [wall * 1e3, cold_total], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        vals = [float(v) for v in tt.cpu()]
        ph = dict(zip(keys, vals[: len(keys)]))
        ph["wall_ms_python_call"] = vals[len(keys)]
        ph["first_call_total_ms"] = vals[len(keys) + 1]
        ph["grm_tflops_aggregate_incl_allreduce"] = n * (n + 1.0) * p / ((ph["grm_ms"] + ph["allreduce_ms"]) * 1e-3) / 1e12
        ph["markers_per_s_whole_gwaslmm"] = p / (ph["total_ms"] * 1e-3)
        ph["lanczos_steps"] = tm["lanczos_steps"]
        ph["launches_this_rank"] = tm["launches"]
        idx = res["idx_cols"]
        ph["markers_kept"] = int(idx.size)
        ph["max_neglog10p"] = float(np.nanmax(res["neglog10p"][idx - 1]))
        ph["sum_abs_z"] = float(np.nansum(np.abs(res["stat"][idx - 1])))  # a checksum to compare across GPU counts
        if storage == "packed":
            ph["pack_s"] = pack_s
        out[storage] = ph
        sm.free()
    if m is not None:
        m.free()
    return out


def run_config3_tetraploid(gbm_b200, _lib, grp, world, rank, hbm_peak):
    """BASELINE configs[3]: grmploidyaware + gwaslmm, tetraploid allele frequencies, n = 2,000 x p = 500,000 -- the
    ploidy-aware branch of gwasprep (/root/reference/src/gwas.jl:117-121: ploidy = Int(round(1 / minimum(G[G .!= 0]))),
    then grmploidyaware) -- sharded over the ranks through gbm_sharded_generate + gbm_sharded_gwas.  Float64 storage
    (FP64 DMMA GRM, Float64 scan) and dosage codes (INT8 GRM, u8 scan).  Parity at this full size:
    tests/test_gpu_fullsize.py::test_config3_tetraploid_full_size."""
    import torch
    import torch.distributed as dist

    from gbm_b200 import multigpu
    from oracle import synth

    n, p, kind = 2_000, 500_000, 1  # KIND_TETRAPLOID
    y = synth.phenotype(SEED, n, p, kind)
    ys = (y - y.mean()) / y.std(ddof=1)
    out = {"workload": f"grmploidyaware + gwaslmm, tetraploid, n={n} p={p} (BASELINE configs[3]), {world} GPU(s)",
           "reference": "gwas.jl:117-121 (ploidy-aware branch), :344-389"}
    keys = ("colstats_ms", "grm_ms", "allreduce_ms", "kstd_pc1_ms", "eig_ms", "scan_ms", "gather_ms", "total_ms", "scan_kernel_ms")
    for storage in ("float64", "packed"):
        sm = multigpu.ShardedMatrix.generate(grp, SEED, n, p, kind, pack=(storage == "packed"))
        if storage == "packed" and not sm.packed:
            sm.free()
            break
        res = None
        for _ in range(2):  # cold, warm
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            res = sm.gwas(ys, model=_lib.MODEL_LMM, grm_type=_lib.GRM_PLOIDY_AWARE, want=("stat", "neglog10p"), out=res)
        tm = res["timing"]
        tt = torch.tensor([tm[k] for k in keys], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ph = dict(zip(keys, (float(v) for v in tt.cpu())))
        p_loc = max(sm.ncols)
        bytes_per = 8.0 if storage == "float64" else 1.0
        scan_gbps = bytes_per * n * p_loc / (ph["scan_kernel_ms"] * 1e-3) / 1e9
        grm_tf = n * (n + 1.0) * p / ((ph["grm_ms"] + ph["allreduce_ms"]) * 1e-3) / 1e12
        idx = res["idx_cols"]
        ph.update(ploidy_inferred=tm["ploidy"], markers_kept=int(idx.size), lanczos_steps=tm["lanczos_steps"],
                  markers_per_s_whole_gwaslmm=p / (ph["total_ms"] * 1e-3),
                  grm_tflops_aggregate_incl_allreduce=grm_tf,
                  max_neglog10p=float(np.nanmax(res["neglog10p"][idx - 1])),
                  sum_abs_z=float(np.nansum(np.abs(res["stat"][idx - 1]))),
                  roofline_scan={"bound": "hbm", "kernel": "scan_sums_kernel<16,2>" if storage == "float64" else "scan_sums_u8_tc_kernel",
                                 "achieved": scan_gbps, "peak": hbm_peak, "unit": "GB/s", "frac": scan_gbps / hbm_peak,
                                 "algorithmic_bytes_per_launch": bytes_per * n * p_loc,
                                 "note": "slowest rank's streaming kernel; its columns are only 2,000 entries (16 KB) long"})
        if storage == "float64":
            ph["roofline_grm"] = {"bound": "tensor", "kernel": "grm_dmma_kernel", "achieved": grm_tf / world, "peak": 40.0,
                                  "unit": "TFLOP/s", "frac": grm_tf / world / 40.0,
                                  "peak_source": "B200 FP64 datasheet (MEASURED_PEAKS.json has no FP64 figure; cuBLAS DGEMM "
                                                 "measured in this run is in grm.cublas_dgemm_8192_tflops)",
                                  "note": "per GPU, n(n+1)p SYRK flops / (contraction + centring passes + all-reduce wall time)"}
        out[storage] = ph
        sm.free()
    return out


def run_config4_stream(args, gbm_b200, _lib, lib, world, rank, j0, barrier):
    """BASELINE configs[4]: gwasols multi-trait batch, 20 traits x n = 20,000 x p = 2,000,000 SNPs streamed from host
    memory (the marker loop /root/reference/src/gwas.jl:239-249 once per trait in the reference; here ONE pass over the
    genotypes for all 20 traits, scan_sums_mt_kernel on the FP64 tensor pipe per column block).  The whole matrix is
    320 GB of Float64; each rank streams a bounded host-resident sample of its share per step through gbm_scan_host
    (PAGEABLE memory) and the full job's time is the extrapolation 2,000,000 / rate.  Float64 copies are PCIe-bound:
    reported as a fraction of the link's plain pinned-copy rate measured in the same run."""
    import ctypes

    import torch
    import torch.distributed as dist

    n, T, p_total = 20_000, 20, 2_000_000
    pe = args.stream_markers
    rng = np.random.default_rng(11)
    Y = np.asfortranarray(rng.normal(size=(n, T)))
    C = rng.normal(size=(n, 1))
    C -= C.mean()
    sub = gbm_b200.DeviceMatrix.generate(SEED, n, pe, KIND_DIPLOID, col0=rank * pe)
    info = sub.info()
    pinned = torch.empty((pe, n), dtype=torch.float64, pin_memory=True)
    cudart = ctypes.CDLL("libcudart.so.12")
    assert cudart.cudaMemcpy(ctypes.c_void_p(pinned.data_ptr()), ctypes.c_void_p(info["device_ptr"]),
                             ctypes.c_size_t(8 * n * pe), ctypes.c_int(2)) == 0
    # the same block resident: device-only rate of the 20-trait kernel at this n
    plan = gbm_b200.ScanPlan(sub, Y, C, model=_lib.MODEL_OLS)
    dstat = torch.empty(pe * T, dtype=torch.float64, device="cuda")
    for _ in range(2):
        plan.run(stat=dstat)
    tm = plan.run(stat=dstat)
    plan.free()
    sub.free()
    del dstat
    host = np.empty((pe, n))
    host[:] = pinned.numpy()
    stat = np.zeros((T, pe))  # p x T column-major
    nlp = np.zeros((T, pe))

    def step(buf, flags):
        _lib.check(lib.gbm_scan_host(_lib.ptr(buf), n, pe, n, _lib.ptr(Y), T, n, _lib.ptr(C), 1, n, _lib.MODEL_OLS, flags,
                                     None, None, _lib.ptr(stat), _lib.ptr(nlp), None, None, None))

    def timed(buf, flags, steps=2):
        step(buf, flags)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            step(buf, flags)
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        ltm = _lib.last_timing()
        rate = pe * world * steps / dt
        return {"markers_per_s": rate, "marker_trait_tests_per_s": rate * T, "estimated_full_job_s": p_total / rate,
                "host_read_gbps_per_gpu": 8.0 * n * pe * steps / dt / 1e9, "h2d_bytes_per_step": ltm["h2d_bytes"],
                "blocks_as_codes": ltm["packed_blocks"]}

    dev = torch.empty((pe, n), dtype=torch.float64, device="cuda")
    dev.copy_(pinned, non_blocking=True)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    dev.copy_(pinned, non_blocking=True)
    ev1.record()
    torch.cuda.synchronize()
    link = 8.0 * n * pe / (ev0.elapsed_time(ev1) * 1e-3) / 1e9
    del dev
    out = {"workload": f"gwasols batch: {T} traits x n={n} x p={p_total} streamed from host memory over {world} GPU(s) "
                       f"(BASELINE configs[4]); sample: {pe} markers per rank per step ({8e-9 * n * pe:.1f} GB of Float64)",
           "resident_block": {"kernel_ms": tm["kernel_ms"], "sums_kernel_ms": tm["main_ms"],
                              "markers_per_s_per_gpu": pe / (tm["kernel_ms"] * 1e-3),
                              "hbm_GBps": 8.0 * n * pe / (tm["main_ms"] * 1e-3) / 1e9,
                              "dmma_tflops": 2.0 * n * pe * 8 * 3 / (tm["main_ms"] * 1e-3) / 1e12},
           "h2d_link_gbps_plain_pinned_copy": link}
    e = timed(host, _lib.SCAN_HOST_NO_PACK)
    e.update(host_memory="pageable", frac_of_link=e["host_read_gbps_per_gpu"] / link,
             roofline={"bound": "pcie", "achieved": e["host_read_gbps_per_gpu"], "peak": link, "unit": "GB/s per GPU",
                       "frac": e["host_read_gbps_per_gpu"] / link, "algorithmic_bytes_per_marker": 8 * n})
    out["float64_copies"] = e
    e = timed(pinned, _lib.SCAN_HOST_NO_PACK)
    e.update(host_memory="pinned", frac_of_link=e["host_read_gbps_per_gpu"] / link)
    out["float64_copies_pinned"] = e
    e = timed(host, 0)
    e.update(host_memory="pageable", note="API default: diploid dosages are packed to 1-byte codes by the host cores / on the device")
    out["default_packing"] = e
    return out


def cpu_whole_function(A, y):
    """The reference's whole gwasols on the host cores, restated with the fastest stock pieces: column std + filter
    (gwas.jl:112-115), GRM through BLAS (the call at :124), K standardisation (:130), PCA by LAPACK SVD (:234), then
    the per-marker loop (:239-249) by the oracle's C/OpenMP twin.  Returns per-phase seconds."""
    from threadpoolctl import threadpool_limits

    from oracle import cbind, gwas_oracle as go

    cores = cbind.use_all_cores()
    t = {}
    with threadpool_limits(limits=cores):
        t0 = time.perf_counter()
        mu, v = cbind.colstats(A)
        t["colstats_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        Z = A - mu[None, :]
        K = (Z @ Z.T) / A.shape[1]
        del Z
        t["grm_blas_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        pc = go.pca_pc1(go.standardise_K(K))
        t["kstd_svd_s"] = time.perf_counter() - t0
    ys = (y - y.mean()) / y.std(ddof=1)
    t0 = time.perf_counter()
    so, sl, keep = cbind.gwasols_raw(A, ys, pc)
    t["marker_loop_s"] = time.perf_counter() - t0
    t["total_s"] = sum(t.values())
    t["cores"] = cores
    return t, sl[keep]


def run_whole_api(gbm_b200, with_cpu=True):
    """The call a user of the reference makes: gwaslmm(genomes = ..., phenomes = ...) -> Fit (gwas.jl:329-337) through
    the host mirror (same keyword API over the C ABI; Genomes holds a pageable host matrix), wall clock per call incl.
    ingestion, filter, GRM, PC1, scan and Fit assembly -- on BASELINE configs[0] (n=300, l=10,000, continuous
    frequencies) and configs[1]'s shape (n=5,000 x p=100,000 diploid).  CPU arm: cpu_whole_function on the same
    matrices."""
    from oracle import synth

    out = {}
    for name, n, p, kind in (("config0_n300_l10000", 300, 10_000, 2), ("config1_shape_n5000_p100000", 5_000, 100_000, 0)):
        A = synth_block_chunked(n, p) if kind == 0 else synth.block(SEED, n, 0, p, kind)
        y = synth.phenotype(SEED, n, p, kind)
        g = gbm_b200.Genomes.from_matrix(A)
        ph = gbm_b200.Phenomes.from_matrix(y, entries=g.entries)
        d = {"n": n, "p": p}
        for fn_name in ("gwasols", "gwaslmm"):
            fn = getattr(gbm_b200, fn_name)
            import gc

            fit = fn(genomes=g, phenomes=ph)  # first call: library / cuSOLVER initialisation
            ts = []
            for _ in range(5 if n <= 1000 else 4):
                gc.collect()  # the harness builds 100,000-element label lists per call: keep the interpreter's
                gc.disable()  # generational collector out of the timed call (it showed up as 0.5-1 s outliers)
                t0 = time.perf_counter()
                fit = fn(genomes=g, phenomes=ph)
                ts.append(time.perf_counter() - t0)
                gc.enable()
            d[fn_name] = {"seconds_per_call_median": float(np.median(ts)), "seconds_per_call_max": float(max(ts)),
                          "markers_per_s": p / float(np.median(ts)), "storage": fit.extras["storage"],
                          "l_kept": int(fit.b_hat.size)}
        if with_cpu:
            t, z_cpu = cpu_whole_function(A, y)
            d["cpu_whole_function"] = dict(t, markers_per_s=p / t["total_s"], kind="port",
                                           note="BLAS GRM + LAPACK SVD + C/OpenMP marker loop on all host cores")
            d["speedup_gwaslmm_vs_cpu_whole_function"] = t["total_s"] / d["gwaslmm"]["seconds_per_call_median"]
            zg = fit.b_hat
            if zg.size == z_cpu.size:
                d["max_abs_diff_z_vs_cpu"] = float(np.max(np.abs(np.abs(zg) - np.abs(z_cpu))))
        out[name] = d
        del A, g, ph
    return out


def run_transform2(gbm_b200, n, l):
    """Pairwise transformation screen (transform2 with f = mult, transformation.jl:319-466): l^2
    regressions y ~ 1 + x_i x_j on a resident n x l matrix.  FP64-pipe-bound: 4 FP64 instructions
    per (pair, row); the roofline is the 64 FP64 instructions / clk / SM of the B200 pipe."""
    from gbm_b200 import _lib, transform as tr

    dm = gbm_b200.DeviceMatrix.generate(SEED, n, l, KIND_DIPLOID)
    rng = np.random.default_rng(5)
    y = rng.normal(size=n)
    out = {"workload": f"transform2(mult) n={n} l={l}: {l * l} regressions (ordered pairs)"}
    for f, name, instr in ((tr.mult, "mult", 4), (tr.addnorm, "addnorm", 5), (tr.raise_, "raise", None)):
        tr.transform2_screen(dm, y, f, 1000)
        t0 = time.perf_counter()
        _, cnt, _ = tr.transform2_screen(dm, y, f, 1000)
        wall = time.perf_counter() - t0
        ms = _lib.last_timing()["main_ms"]
        d = {"pair_kernel_ms": ms, "regressions_per_s": l * l / (ms * 1e-3), "wall_s_with_selection": wall,
             "selected": int(cnt.size)}
        if instr:
            info = _lib.device_info()
            per_clk = instr * float(l) * l * n / (ms * 1e-3) / (info["sm_count"] * 1.965e9)
            d["fp64_instr_per_clk_per_sm"] = per_clk
            d["frac_of_fp64_pipe"] = per_clk / 64.0
        out[name] = d
    dm.free()
    return out


def run_lmm(gbm_b200, _lib, n, pm):
    """GRM-covariance LMM engine (model of gwasreml): GRM on the sample, syevd (cuSOLVER, timed
    separately), rotation U'A by the DMMA GEMM, per-marker REML delta search."""
    import torch

    out = {"n": n, "markers": pm}
    dm = gbm_b200.DeviceMatrix.generate(SEED, n, pm, KIND_DIPLOID)
    dK = torch.empty(n * n, dtype=torch.float64, device="cuda")
    dm.grm(_lib.GRM_SIMPLE, 2, 0, out=dK)
    # polygenic phenotype (h2 = 0.5) so that delta is interior: y = g + e with g ~ N(0, K)-like
    rng = np.random.default_rng(3)
    cols = rng.choice(pm, size=min(pm, 2000), replace=False)
    g = np.zeros(n)
    for j in cols:
        c = dm.download(int(j), 1)[:, 0]
        g += rng.normal() * (c - c.mean())
    g /= g.std()
    y = np.sqrt(0.5) * g + np.sqrt(0.5) * rng.normal(size=n)
    t0 = time.perf_counter()
    plan = gbm_b200.LmmPlan(dK, y)
    out["plan_create_s"] = time.perf_counter() - t0
    out["cusolver_syevd_s"] = plan.eig_ms * 1e-3
    out["null_log_delta"] = plan.null_log_delta
    plan.run(dm)  # warm-up
    t0 = time.perf_counter()
    res = plan.run(dm)
    out["run_s"] = time.perf_counter() - t0
    out["rotation_gemm_tflops"] = res["gemm_tflops"]
    out["rotation_gemm_ms"] = res["timing"]["main_ms"]
    out["delta_search_ms"] = res["search_ms"]
    out["markers_per_s"] = pm / out["run_s"]
    ld = res["log_delta"]
    out["log_delta_range"] = [float(np.nanmin(ld)), float(np.nanmax(ld))]
    out["max_neglog10p"] = float(np.nanmax(res["neglog10p"]))
    plan.free()
    dm.free()
    return out


if __name__ == "__main__":
    sys.exit(main())
