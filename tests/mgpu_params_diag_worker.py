"""torchrun worker for tests/test_gpu_params_diag.py: a D = 256 diagonal Gaussian fit() sharded over the ranks with the
parameter step on the device.  Every rank draws its parameters from the same all-reduced statistics with the same
counter-based streams, so get_params_diag must return the same bytes on every rank."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import dpmm_pkg  # noqa: E402
from tests.diag_util import axis_aligned_data  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
pkg = dpmm_pkg.load()
from dpmmsubclusters_jl_b200 import host as H, priors as P  # noqa: E402

D = 256
hyper = P.diag_niw_hyperparams(1.0, np.zeros(D), 10.0, np.ones(D))
x, z = axis_aligned_data(40_000, D, 12, 5, hyper)
n = x.shape[1]
lo, hi = rank * n // world, (rank + 1) * n // world
ids = [pkg.GpuSweep.nccl_unique_id() if rank == 0 else None]
dist.broadcast_object_list(ids, src=0)
out = pkg.fit(x[:, lo:hi], hyper, 10.0, iters=40, seed=11, burnout=10, device=local, device_params=True,
              shard=(lo, n), comm=(ids[0], rank, world))
sw = out[-1].group.sweep
K = len(out[1])
params = sw.get_params_diag(K)
blob = b"".join(a.tobytes() for a in params)
gathered = [None] * world
dist.all_gather_object(gathered, (K, blob, lo, sw.get_labels()))
if rank == 0:
    assert all(g[0] == K for g in gathered), [g[0] for g in gathered]
    assert all(g[1] == blob for g in gathered), "ranks hold different parameters"
    labels = np.concatenate([g[3] for g in sorted(gathered, key=lambda g: g[2])])
    nmi = H.normalized_mutual_info(z, labels)
    assert nmi >= 0.9, nmi
    print("MGPU_PARAMS_DIAG_OK", K, f"{nmi:.4f}", len(blob), flush=True)
dist.barrier()
dist.destroy_process_group()
