"""torchrun worker for tests/test_gpu_outlier.py: a D = 2 NIW fit() with the outlier component, sharded over the ranks
with the parameter step on the device.  Every rank must hold the same parameters and weights (cluster 1 included)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import dpmm_pkg  # noqa: E402
from tests.test_outlier_host import background_data, OUTLIER, PRIOR  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
pkg = dpmm_pkg.load()
from dpmmsubclusters_jl_b200 import host as H  # noqa: E402

x, gt = background_data(1)
rng = np.random.default_rng(0)
perm = rng.permutation(x.shape[1])          # background points on every rank
x, gt = x[:, perm], gt[perm]
n = x.shape[1]
lo, hi = rank * n // world, (rank + 1) * n // world
ids = [pkg.GpuSweep.nccl_unique_id() if rank == 0 else None]
dist.broadcast_object_list(ids, src=0)
out = pkg.fit(x[:, lo:hi], PRIOR, 10.0, iters=150, seed=11, device=local, device_params=True, outlier_weight=0.05,
              outlier_params=OUTLIER, shard=(lo, n), comm=(ids[0], rank, world))
sw = out[-1].group.sweep
K = len(out[1])
params = sw.get_params_niw(K)
blob = b"".join(a.tobytes() for a in params)
gathered = [None] * world
dist.all_gather_object(gathered, (K, blob, lo, sw.get_labels()))
if rank == 0:
    assert all(g[0] == K for g in gathered), [g[0] for g in gathered]
    assert all(g[1] == blob for g in gathered), "ranks hold different parameters"
    assert params[3][0] == np.float32(0.05)
    labels = np.concatenate([g[3] for g in sorted(gathered, key=lambda g: g[2])])
    cap = (labels[gt == 0] == 1).mean()
    assert cap >= 0.8, cap
    print("MGPU_OUTLIER_OK", K, f"{cap:.3f}", flush=True)
dist.barrier()
dist.destroy_process_group()
