"""Per-stage device times of diagonal Gaussian sweeps (DPMM_PRIOR_DIAG_GAUSSIAN) at four shapes, and fit() iterations
per second with the parameter step on the device and on the host, one JSON line per measurement on stdout and in
profiles/diag_bench.jsonl.

    python tools/bench_diag.py [--shapes G1,G2,G3,G4] [--sweeps 20] [--warmup 3] [--fit-shapes G1,G2,G3]
                               [--fit-iters 40] [--fit-reps 2]

fit() runs from one cluster on data drawn like the sweep shapes', the two paths alternated --fit-reps times each; it
reports iterations per second inside the loop and for the whole call.  One more fit per path runs with kernel timing
on and reports the `params` kernel time per iteration (the device parameter step and the packing of the parameter
images; on the host path only the packing).

Stage times come from dpmm_timing_read (CUDA events around each kernel), after the warm-up sweeps.  Each stage's
share is of the larger of its two bounds, computed from the shapes here:
  label     4 n K D flop (two FMAs per point, cluster and feature) at bench.FFMA2_PEAK_TFLOPS; 4 n D bytes (one pass
            over X) at bench's HBM figure
  sub-label 8 n D flop (two distributions); 4 n D bytes
  sort      8 n bytes (labels in, permutation out)
  stats     4 n D bytes
Every X is larger than L2.  The card's name and power limit are printed with the numbers."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"G1": (1_000_000, 128, 20), "G2": (1_000_000, 512, 50), "G3": (200_000, 4096, 20), "G4": (100_000, 16384, 100)}


def device_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def make_data(n, D, K, seed):
    """Axis-aligned clusters generated on the device, returned as an n x D host array (= D x n column-major), with the
    true means and variances."""
    import torch
    gen = torch.Generator(device="cuda").manual_seed(seed)
    means = torch.randn(K, D, device="cuda", generator=gen) * 10
    sd = torch.rand(K, D, device="cuda", generator=gen) + 0.5
    z = torch.randint(0, K, (n,), device="cuda", generator=gen)
    x = np.empty((n, D), np.float32)
    step = max(1, (1 << 28) // D)
    for i in range(0, n, step):
        zz = z[i:i + step]
        x[i:i + step] = (means[zz] + sd[zz] * torch.randn(len(zz), D, device="cuda", generator=gen)).cpu().numpy()
    return x, means.cpu().numpy().astype(np.float64), (sd.cpu().numpy().astype(np.float64)) ** 2


def run_shape(pkg, tag, n, D, K, sweeps, warmup, ffma_tflops, hbm_gbs):
    x, means, var = make_data(n, D, K, D + K)
    rng = np.random.default_rng(K)
    mu = (means[:, None, :] + 0.3 * rng.standard_normal((K, 3, D))).astype(np.float32)
    vv = (var[:, None, :] * rng.uniform(0.8, 1.25, (K, 3, D))).astype(np.float32)
    ld = np.log(vv.astype(np.float64)).sum(-1).astype(np.float32)
    w = rng.dirichlet(np.ones(K) * 5).astype(np.float32)
    lr = rng.dirichlet(np.ones(2) * 5, size=K).astype(np.float32)
    g = pkg.GpuSweep(x.T, pkg.DIAG, seed=1)
    del x
    g.init_labels(K)
    g.set_params_diag(mu, vv, ld, w, lr)

    def sweep():
        g.sample_labels(False)
        g.sample_sublabels()
        g.suff_stats(fetch=False)

    for _ in range(warmup):
        sweep()
    g.sync()
    t0 = time.perf_counter()
    for _ in range(sweeps):
        sweep()
    g.sync()
    wall = time.perf_counter() - t0
    g.timing_enable(True)
    g.timing_read(reset=True)
    for _ in range(sweeps):
        sweep()
    tm = g.timing_read(reset=True)
    g.timing_enable(False)
    g.close()
    ms = {k: tm[k][0] / sweeps for k in ("label", "sort", "sublabel", "stats", "stats_aux")}
    xb = 4.0 * n * D
    bounds = {"label": (4.0 * n * K * D, xb), "sublabel": (8.0 * n * D, xb), "sort": (0.0, 8.0 * n), "stats": (0.0, xb)}
    share = {}
    for k, (fl, by) in bounds.items():
        tf, th = fl / (ffma_tflops * 1e12) * 1e3, by / (hbm_gbs * 1e9) * 1e3
        share[k] = dict(bound="ffma" if tf >= th else "hbm", floor_ms=max(tf, th), share=max(tf, th) / ms[k] if ms[k] > 0 else None)
    return dict(shape=tag, n=n, D=D, K=K, sweeps=sweeps, stage_ms=ms, sweep_ms_events=sum(ms.values()),
                sweeps_per_s=sweeps / wall, share_of_bound=share,
                label_tflops=4.0 * n * K * D / (ms["label"] * 1e-3) / 1e12)


def run_fit(pkg, tag, iters, reps):
    from dpmmsubclusters_jl_b200 import priors as P
    n, D, K = SHAPES[tag]
    x, _, _ = make_data(n, D, K, 7)
    xt = x.T
    hyper = P.diag_niw_hyperparams(1.0, np.zeros(D), 10.0, np.ones(D))
    made = []

    def factory(timing):
        def make(xx, kind, seed, goff):
            g = pkg.GpuSweep(xx, kind, seed=seed, global_offset=goff)
            g.timing_enable(timing)
            made.append(g)
            return g
        return make

    def one(dev, timing):
        made.clear()
        t0 = time.perf_counter()
        _, clusters, _, iter_count, *_ = pkg.fit(xt, hyper, 10.0, iters=iters, seed=1, burnout=10, device_params=dev,
                                                 sweep_factory=factory(timing))
        made[0].sync()
        wall = time.perf_counter() - t0
        params_ms = made[0].timing_read(reset=True)["params"][0] / len(iter_count) if timing else None
        return len(clusters), len(iter_count) / float(np.sum(iter_count)), len(iter_count) / wall, params_ms

    recs = {dev: dict(shape=f"{tag}-fit", path="device" if dev else "host", n=n, D=D, K_true=K, init_clusters=1,
                      iters=iters, loop_iters_per_s=[], call_iters_per_s=[], K_final=[]) for dev in (True, False)}
    for _ in range(reps):
        for dev in (True, False):
            kf, loop, call, _ = one(dev, False)
            recs[dev]["loop_iters_per_s"].append(loop)
            recs[dev]["call_iters_per_s"].append(call)
            recs[dev]["K_final"].append(kf)
    for dev in (True, False):
        recs[dev]["params_kernel_ms_per_iter"] = one(dev, True)[3]
    return [recs[True], recs[False]]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="G1,G2,G3,G4")
    ap.add_argument("--sweeps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--fit-shapes", default="G1,G2,G3")
    ap.add_argument("--fit-iters", type=int, default=40)
    ap.add_argument("--fit-reps", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "diag_bench.jsonl"))
    args = ap.parse_args()
    import bench
    import __graft_entry__
    __graft_entry__.build()
    import dpmm_pkg
    pkg = dpmm_pkg.load()
    hbm_gbs = bench.peaks()["hbm_gbs"]
    name, power = device_info()
    print(f"device: {name}; power limit, max SM clock: {power}", flush=True)
    recs = []
    for tag in args.shapes.split(","):
        n, D, K = SHAPES[tag]
        recs.append(run_shape(pkg, tag, n, D, K, args.sweeps, args.warmup, bench.FFMA2_PEAK_TFLOPS, hbm_gbs))
    if args.fit_iters > 0:
        for tag in filter(None, args.fit_shapes.split(",")):
            recs.extend(run_fit(pkg, tag, args.fit_iters, args.fit_reps))
    with open(args.out, "w") as f:
        for r in recs:
            r.update(device=name, power_limit_and_max_sm_clock=power, ffma2_peak_tflops=bench.FFMA2_PEAK_TFLOPS, hbm_gbs=hbm_gbs)
            print(json.dumps(r), flush=True)
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
