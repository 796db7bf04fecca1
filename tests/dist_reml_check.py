"""Multi-GPU check of the sharded rotation LMM (gwasreml), one process per GPU under torchrun on N GPUs of one box;
collected by pytest through tests/test_gpu_group_reml.py::test_gwasreml_one_process_per_gpu_under_torchrun (marker
`multigpu`), or by hand:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29533 tests/dist_reml_check.py

The library's RANK group (gbm_group_create_rank; torch.distributed only hands out the 128-byte NCCL id): per-rank
column blocks generated on the device, then the one-call gbm_sharded_gwasreml (GRM all-reduce, eigendecomposition on
rank 0 and its broadcast, rotation + delta search per rank, gather) and the plan with a given K, both compared on
rank 0 with the CPU oracle."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "genomicbreedingmodels.jl_b200"))

import numpy as np
import torch
import torch.distributed as dist

import gbm_b200
from gbm_b200 import _lib, multigpu
from oracle import gwas_oracle as go, lmm_oracle as lo, synth


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    gbm_b200.init(local)
    grp = multigpu.Group.from_torch_distributed()
    n, p, seed, kind = 384, 3001, 19, synth.KIND_TETRAPLOID
    A = synth.block(seed, n, 0, p, kind)
    y = synth.phenotype(seed, n, p, kind)
    ys = (y - y.mean()) / y.std(ddof=1)
    K = go.grm_ploidy_aware(A, 4)
    sm = multigpu.ShardedMatrix.generate(grp, seed, n, p, kind, pack=True)
    one = sm.gwasreml(ys, grm_type=_lib.GRM_PLOIDY_AWARE)
    plan = sm.lmm_plan(K, ys)
    res = plan.run()
    plan.free()
    sm.free()
    if rank == 0:
        ref = lo.lmm_scan(A, ys, K)
        keep = ref["keep"]
        zs = max(1.0, np.abs(ref["z"][keep]).max())
        e_1 = np.max(np.abs(one["stat"][keep] - ref["z"][keep])) / zs
        e_p = np.max(np.abs(res["stat"][keep] - ref["z"][keep])) / zs
        e_l = np.max(np.abs(one["log_delta"][keep] - ref["log_delta"][keep]))
        idx_ok = np.array_equal(one["idx_cols"], np.flatnonzero(keep) + 1)
        ok = (idx_ok and e_1 < 1e-9 and e_p < 1e-9 and e_l < 1e-7 and one["timing"]["ploidy"] == 4
              and one["timing"]["n_gpus"] == world)
        print(f"dist_reml_check world={world}: idx_cols equal={idx_ok} one-call z err={e_1:.2e} plan z err={e_p:.2e} "
              f"log delta err={e_l:.2e} | eig {one['timing']['eig_ms']:.1f} ms, broadcast "
              f"{one['timing']['broadcast_ms']:.1f} ms -> {'OK' if ok else 'FAIL'}", flush=True)
        if not ok:
            sys.exit(1)
    grp.free()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
