"""Two-rank check of the device-side posterior summaries, one process per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29547 tests/multi_gpu_posterior_check.py

c2 with device deviates on ring-partitioned ranks.  Nothing of dang_gpu_posterior_* crosses ranks: each rank
accumulates every posterior kind over its own pixels, and its accumulators must equal the numpy restatement of the
update rule over its slice of the states the existing getters download.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import torch
    import torch.distributed as dist

    from dang_b200.engine import Engine, setup_torch_comm
    from dang_b200.healpix import ring_partition
    from helpers import small_case
    from test_gpu_posterior import POST_ALL, _kinds_of, _state, welford

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    nside = int(os.environ.get("DANG_MGC_NSIDE", "16"))
    cfg, sky = small_case("c2", nside, perturb=False)
    bounds = ring_partition(cfg.nside, world, weights=(sky.mask != 0).astype(np.float64))
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    eng = Engine(cfg, sky, device=local, pix_range=(lo, hi))
    setup_torch_comm(eng, mailboxes=os.environ.get("DANG_GPU_MAILBOX", "1") != "0")
    kinds = _kinds_of(cfg)
    eng.posterior_begin(POST_ALL)
    states = []
    for it in range(1, 6):
        eng.gibbs_iteration(it, seed=9)
        eng.posterior_accumulate()
        states.append(_state(eng, kinds))
    for key in kinds:
        mean, std, n = eng.posterior(*key)
        want_mean, _, want_std = welford([s[key][..., lo:hi] for s in states])
        assert n == 5 and np.array_equal(mean[..., lo:hi], want_mean), (rank, key)
        assert np.array_equal(std[..., lo:hi], want_std, equal_nan=True), (rank, key)
    eng.comm_check()
    eng.close()
    dist.barrier()
    print(f"rank {rank}/{world}: multi-GPU posterior ok (pixels [{lo},{hi}))", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
