"""fit() with and without the outlier component on the device parameter path: N = 1e6 points of D = 32 from K = 20
Gaussians plus 5 % uniform background over their bounding box.  The two configurations alternate three times in one
process; one JSON line per run goes to --out, preceded by a line with the card's name, power limit and max SM clock.

Per run: iterations/s in the loop (sum of group_step times) and for the whole call, final K, the share of background
points labelled 1 (with the component) and the inlier NMI.  A separate instrumented run per configuration counts the
label launches that took the tensor-core kernel (each is followed by its overflow kernel) against all label launches:
the adaptive switch sends calls to the FMA kernel while the tensor-core kernel finds too many candidate clusters.

    python tools/fit_outlier.py --out profiles/outlier_fit.jsonl
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import dpmm_pkg  # noqa: E402

pkg = dpmm_pkg.load()
from dpmmsubclusters_jl_b200 import host as H, priors as P  # noqa: E402


def data(n, D, K, frac, seed):
    rng = np.random.default_rng(seed)
    x, z, _, _ = pkg.generate_gaussian_data(n, D, K, 100.0, rng)
    lo, hi = x.min(1), x.max(1)
    nb = int(round(n * frac / (1 - frac)))
    b = rng.uniform(lo[:, None], hi[:, None], (D, nb)).astype(np.float32)
    bg = np.concatenate([np.zeros(n, bool), np.ones(nb, bool)])
    out = P.niw_hyperparams(1.0, (lo + hi) / 2.0, D + 3.0, np.diag((hi - lo) ** 2 / 12.0))
    return np.concatenate([x, b], 1), np.concatenate([z.astype(np.int64), np.zeros(nb, np.int64)]), bg, out


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"card": name, "power_limit": power, "max_sm_clock": clock}


def run(x, z, bg, hyper, out, outlier, iters, seed, timing=False):
    sweeps = []

    def factory(xx, kind, sd, goff):
        sw = pkg.GpuSweep(xx, kind, seed=sd, global_offset=goff)
        if timing:
            sw.timing_enable(True)
        sweeps.append(sw)
        return sw
    kw = dict(outlier_weight=0.05, outlier_params=out) if outlier else {}
    t0 = time.perf_counter()
    labels, _, weights, iter_count, *_ = pkg.fit(x, hyper, 10.0, iters=iters, seed=seed, device_params=True,
                                                 sweep_factory=factory, **kw)
    wall = time.perf_counter() - t0
    r = {"outlier": outlier, "seed": seed, "iters": iters, "final_K": len(weights),
         "loop_it_per_s": round(len(iter_count) / sum(iter_count), 2), "call_it_per_s": round(iters / wall, 2),
         "background_in_1": round(float((labels[bg] == 1).mean()), 4),
         "inliers_in_1": round(float((labels[~bg] == 1).mean()), 5),
         "inlier_nmi": round(H.normalized_mutual_info(z[~bg], labels[~bg]), 4)}
    if timing:
        t = sweeps[0].timing_read()
        r = {"outlier": outlier, "seed": seed, "label_launches": t["label"][1],
             "tensor_core_label_launches": t["label_ovf"][1]}
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n", type=float, default=1e6)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    D, K = 32, 20
    x, z, bg, out = data(int(a.n), D, K, 0.05, 0)
    hyper = P.niw_hyperparams(1.0, np.zeros(D), D + 3.0, np.eye(D))
    lines = [dict(card(), n=int(x.shape[1]), D=D, K_true=K, background_frac=0.05)]
    run(x, z, bg, hyper, out, True, 5, 99)                      # warm-up: module load, first allocations
    for rep in range(a.reps):
        for outlier in (False, True):
            lines.append(run(x, z, bg, hyper, out, outlier, a.iters, 1 + rep))
            print(json.dumps(lines[-1]), flush=True)
    for outlier in (False, True):
        lines.append(run(x, z, bg, hyper, out, outlier, a.iters, 1, timing=True))
        print(json.dumps(lines[-1]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
