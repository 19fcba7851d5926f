"""fit() on the C3 workload (multinomial, N = 1e6, D = 100, K = 20) with the parameter step on the device and on the
host, alternated: whole-call and in-loop iterations/s, final K and NMI, and the per-iteration GPU time of the
parameter-step kernels (dpmm_timing_read, kind "params").  Prints the card and its power limit with the numbers.

    python tools/fit_mnm.py [--reps 3] [--iters 100] [--n 1000000]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
        name, power, clock = (s.strip() for s in q.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except (OSError, subprocess.CalledProcessError, IndexError, ValueError):
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown", "max_sm_clock": "unknown"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--n", type=int, default=10 ** 6)
    args = ap.parse_args()
    import __graft_entry__ as ge
    ge.build()
    import dpmm_pkg
    pkg = dpmm_pkg.load()
    from dpmmsubclusters_jl_b200.host import normalized_mutual_info
    x, z, _ = pkg.generate_mnmm_data(args.n, 100, 20, 50, np.random.default_rng(0))
    hyper = pkg.multinomial_hyper(np.ones(100, np.float32))
    timed = []

    def factory(xx, kind, seed, goff):
        sw = pkg.GpuSweep(xx, kind, seed=seed, global_offset=goff)
        if timed:
            sw.timing_enable(True)
        return sw

    def run(device_params):
        t0 = time.perf_counter()
        out = pkg.fit(x, hyper, 10.0, iters=args.iters, seed=1, burnout=20, device_params=device_params,
                      sweep_factory=factory)
        wall = time.perf_counter() - t0
        r = {"device_params": device_params, "iters_per_s": args.iters / wall,
             "loop_iters_per_s": args.iters / float(sum(out[3])), "final_K": len(out[1]),
             "nmi": round(normalized_mutual_info(z, out[0]), 4)}
        if timed:
            ms, cnt = out[-1].group.sweep.timing_read()["params"]
            r["params_kernel_ms_per_iter"] = ms / args.iters
            r["params_launches_per_iter"] = cnt / args.iters
        out[-1].group.sweep.close()
        return r

    for mode in (True, False):                # first calls: CUDA module loading and first launches
        run(mode)
    results = [run(mode) for _ in range(args.reps) for mode in (True, False)]
    timed.append(True)                        # kernel timing in runs of their own: the events cost host time
    results += [run(mode) for mode in (True, False)]
    print(json.dumps({"card": card(), "workload": f"C3 multinomial N={args.n} D=100 K=20, alpha=10, prior alpha=1, "
                      f"{args.iters} iterations, burnout 20, seed 1", "runs": results}, indent=1), flush=True)


if __name__ == "__main__":
    main()
