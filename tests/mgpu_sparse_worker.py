"""torchrun worker for tests/test_gpu_mnm_sparse.py: a D = 3000 sparse multinomial model sharded over the ranks; the
all-reduced statistics and the gathered labels / sub-labels must equal a one-GPU dense run of the whole matrix."""
import os
import sys

import numpy as np
import scipy.sparse as sps
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import dpmm_pkg  # noqa: E402
from tests.util import make_mnm_case, set_params  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
pkg = dpmm_pkg.load()
case = make_mnm_case(3000, 24, 20000, seed=8, trials=20)
x = case["x"]
n = case["n"]
lo, hi = rank * n // world, (rank + 1) * n // world
g = pkg.GpuSweep(sps.csc_matrix(x[:, lo:hi]), pkg.MULTINOMIAL, seed=42, global_offset=lo, device=local)
ids = [pkg.GpuSweep.nccl_unique_id() if rank == 0 else None]
dist.broadcast_object_list(ids, src=0)
g.comm_init(ids[0], rank, world)
set_params(g, case)
g.sample_labels(False)
g.sample_sublabels()
counts, sx, _ = g.suff_stats()
gathered = [None] * world
dist.all_gather_object(gathered, (lo, g.get_labels(), g.get_sublabels()))
if rank == 0:
    ref = pkg.GpuSweep(x, pkg.MULTINOMIAL, seed=42, global_offset=0, device=local)
    set_params(ref, case)
    ref.sample_labels(False)
    ref.sample_sublabels()
    rc, rsx, _ = ref.suff_stats()
    np.testing.assert_array_equal(np.concatenate([t[1] for t in sorted(gathered, key=lambda t: t[0])]), ref.get_labels())
    np.testing.assert_array_equal(np.concatenate([t[2] for t in sorted(gathered, key=lambda t: t[0])]), ref.get_sublabels())
    np.testing.assert_array_equal(counts, rc)
    np.testing.assert_array_equal(sx, rsx)
    ref.close()
    print("MGPU_SPARSE_OK", counts[:, 0].sum(), flush=True)
g.close()
dist.barrier()
dist.destroy_process_group()
