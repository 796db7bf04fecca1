"""gwasreml at the project's target size (BASELINE configs[2]: n = 10,000 x p = 1,000,000 diploid markers, one trait,
GRM eigen-rotation) through the one-call gbm_sharded_gwasreml on local groups of 1, 2, 4 and 8 GPUs -- those the box
has.  The genotypes are made on the device (gbm_sharded_generate), stored as Float64 and as one-byte dosage codes.
Per group size and storage: one warm-up call, then --reps timed calls; the fastest is reported.

Writes one JSON file per group size, `<out>/r03_reml_group_n<N>.json`, with every gbm_reml_timing field of that call,
markers/s (rotation + search, and the whole call), the rotation's TFLOP/s per GPU and aggregate against a sustained
cuBLAS DGEMM measured in the same run (float64 torch.matmul 8192^3 for >= 1 s), speed-ups over N = 1, sum |z| and
max -log10 p, and the GPU's name, power limit and maximum SM clock (nvidia-smi, read-only query).

    python tools/bench_reml_group.py --out DIR
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "genomicbreedingmodels.jl_b200"))

import numpy as np  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()
    name, power, clock = (s.strip() for s in q[0].split(","))
    return {"gpu": name, "power_limit": power, "clocks_max_sm": clock, "visible_gpus": len(q)}


def sustained_dgemm_tflops(min_s=1.0):
    import torch

    a = torch.randn(8192, 8192, dtype=torch.float64, device="cuda")
    b = torch.randn(8192, 8192, dtype=torch.float64, device="cuda")
    c = torch.matmul(a, b)  # warm-up: cuBLAS picks its kernel
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters, t0 = 0, time.perf_counter()
    e0.record()
    while time.perf_counter() - t0 < min_s:
        for _ in range(4):
            torch.matmul(a, b, out=c)
        iters += 4
        torch.cuda.synchronize()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    del a, b, c
    torch.cuda.empty_cache()
    return 2.0 * 8192 ** 3 * iters / (ms * 1e-3) / 1e12, ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n", type=int, default=10_000)
    ap.add_argument("--p", type=int, default=1_000_000)
    ap.add_argument("--groups", default="1,2,4,8")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--seed", type=int, default=2026)
    a = ap.parse_args()

    import gbm_b200
    from gbm_b200 import _lib, multigpu
    from oracle import synth

    info = gpu_info()
    gbm_b200.init(0)
    dgemm, dgemm_ms = sustained_dgemm_tflops()
    n, p = a.n, a.p
    y = synth.phenotype(a.seed, n, p, synth.KIND_DIPLOID)
    ys = (y - y.mean()) / y.std(ddof=1)
    os.makedirs(a.out, exist_ok=True)
    base = {}
    for N in [int(s) for s in a.groups.split(",")]:
        if N > info["visible_gpus"]:
            print(f"N={N}: not measured ({info['visible_gpus']} GPU(s) visible)", flush=True)
            continue
        grp = multigpu.Group.local(N)
        rec = dict(info, config="BASELINE configs[2]: gwasreml n x p diploid, 1 trait, GRM eigen-rotation",
                   entry_point="gbm_sharded_gwasreml", n=n, p=p, n_gpus=N, reps=a.reps, seed=a.seed,
                   dgemm_sustained_tflops=dgemm, dgemm_window_ms=dgemm_ms, storage={})
        for storage in ("float64", "codes"):
            sm = multigpu.ShardedMatrix.generate(grp, a.seed, n, p, synth.KIND_DIPLOID, pack=storage == "codes")
            assert sm.packed == (storage == "codes")
            sm.gwasreml(ys)  # warm-up
            best = None
            for _ in range(a.reps):
                res = sm.gwasreml(ys)
                if best is None or res["timing"]["total_ms"] < best["timing"]["total_ms"]:
                    best = res
            sm.free()
            tm = best["timing"]
            rs_ms = tm["rotation_ms"] + tm["search_ms"]
            r = dict(timing=tm, markers_per_s_rotation_search=p / (rs_ms * 1e-3), markers_per_s_call=p / (tm["total_ms"] * 1e-3),
                     rotation_tflops_aggregate=tm["rotation_tflops"], rotation_tflops_per_gpu=tm["rotation_tflops"] / N,
                     rotation_per_gpu_over_dgemm=tm["rotation_tflops"] / N / dgemm,
                     sum_abs_z=float(np.nansum(np.abs(best["stat"]))), max_neglog10p=float(np.nanmax(best["neglog10p"])),
                     n_keep=int(best["idx_cols"].size))
            if N == 1:
                base[storage] = (rs_ms, tm["total_ms"])
            if storage in base:
                r["speedup_vs_1_rotation_search"] = base[storage][0] / rs_ms
                r["speedup_vs_1_call"] = base[storage][1] / tm["total_ms"]
            rec["storage"][storage] = r
            print(f"N={N} {storage}: total {tm['total_ms']:.0f} ms (colstats {tm['colstats_ms']:.0f}, GRM {tm['grm_ms']:.0f} "
                  f"+ all-reduce {tm['allreduce_ms']:.0f}, eig {tm['eig_ms']:.0f}, broadcast {tm['broadcast_ms']:.0f}, marker "
                  f"loop {tm['scan_ms']:.0f}, gather {tm['gather_ms']:.0f}); rotation {tm['rotation_ms']:.0f} ms = "
                  f"{tm['rotation_tflops']:.1f} TF aggregate ({r['rotation_per_gpu_over_dgemm']:.2f} of DGEMM {dgemm:.1f} TF "
                  f"per GPU), search {tm['search_ms']:.0f} ms; sum|z| {r['sum_abs_z']:.10e}", flush=True)
        grp.free()
        with open(os.path.join(a.out, f"r03_reml_group_n{N}.json"), "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
