"""torchrun worker for tests/test_gpu_diag.py: a D = 1 000 diagonal Gaussian model sharded over the ranks; the labels
and sub-labels must equal those of the whole data set on one GPU, and the all-reduced statistics its statistics (Float64
sums in another order: to rounding)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import dpmm_pkg  # noqa: E402
from tests.diag_util import make_diag_case, set_params_diag  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
pkg = dpmm_pkg.load()
case = make_diag_case(1000, 24, 20000, seed=8)
n = case["n"]
lo, hi = rank * n // world, (rank + 1) * n // world
g = pkg.GpuSweep(case["x"][:, lo:hi], pkg.DIAG, seed=42, global_offset=lo, device=local)
ids = [pkg.GpuSweep.nccl_unique_id() if rank == 0 else None]
dist.broadcast_object_list(ids, src=0)
g.comm_init(ids[0], rank, world)
set_params_diag(g, case)
g.sample_labels(False)
g.sample_sublabels()
counts, sx, sxx = g.suff_stats()
gathered = [None] * world
dist.all_gather_object(gathered, (lo, g.get_labels(), g.get_sublabels()))
if rank == 0:
    ref = pkg.GpuSweep(case["x"], pkg.DIAG, seed=42, global_offset=0, device=local)
    set_params_diag(ref, case)
    ref.sample_labels(False)
    ref.sample_sublabels()
    rc, rsx, rsxx = ref.suff_stats()
    np.testing.assert_array_equal(np.concatenate([t[1] for t in sorted(gathered, key=lambda t: t[0])]), ref.get_labels())
    np.testing.assert_array_equal(np.concatenate([t[2] for t in sorted(gathered, key=lambda t: t[0])]), ref.get_sublabels())
    np.testing.assert_array_equal(counts, rc)
    np.testing.assert_allclose(sx, rsx, rtol=1e-12, atol=1e-9)
    np.testing.assert_allclose(sxx, rsxx, rtol=1e-12)
    ref.close()
    print("MGPU_DIAG_OK", counts[:, 0].sum(), flush=True)
g.close()
dist.barrier()
dist.destroy_process_group()
