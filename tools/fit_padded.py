"""fit() on Gaussian data at feature widths without NIW kernels of their own (D = 20 and 50: the context runs
zero-padded to 24 and 64), with the parameter step on the device and on the host, alternated: whole-call and
in-loop iterations/s, final K and NMI.  N = 1e6, K_true = 20, fit(x, 10.0) defaults otherwise.  Prints the card
and its power limit with the numbers (and writes them to --out if given).

    python tools/fit_padded.py [--reps 2] [--iters 100] [--n 1000000] [--dims 20,50] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from fit_mnm import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--n", type=int, default=10 ** 6)
    ap.add_argument("--dims", default="20,50")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import __graft_entry__ as ge
    ge.build()
    import dpmm_pkg
    pkg = dpmm_pkg.load()
    from dpmmsubclusters_jl_b200.host import normalized_mutual_info
    info = card()
    results = []
    for D in (int(d) for d in args.dims.split(",")):
        x, z, _, _ = pkg.generate_gaussian_data(args.n, D, 20, 100.0, np.random.default_rng(0))

        def run(device_params):
            t0 = time.perf_counter()
            out = pkg.fit(x, 10.0, iters=args.iters, seed=1, burnout=20, device_params=device_params)
            wall = time.perf_counter() - t0
            out[-1].group.sweep.close()
            return {"D": D, "device_params": device_params, "iters_per_s": args.iters / wall,
                    "loop_iters_per_s": args.iters / float(sum(out[3])), "final_K": len(out[1]),
                    "nmi": round(normalized_mutual_info(z, out[0]), 4)}

        for mode in (True, False):            # first calls: CUDA module loading and first launches
            run(mode)
        for _ in range(args.reps):
            for mode in (True, False):
                results.append(run(mode))
                print(json.dumps(results[-1]), file=sys.stderr, flush=True)
    doc = {"card": info, "workload": f"NIW fit(x, 10.0), N={args.n}, K_true=20, generate_gaussian_data(var 100), "
           f"{args.iters} iterations, burnout 20, seed 1", "runs": results}
    print(json.dumps(doc, indent=1), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
