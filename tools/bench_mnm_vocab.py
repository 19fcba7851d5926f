"""Per-stage device times of multinomial sweeps on large vocabularies (the streaming label kernel, the staged sub-label
kernel and the sliced statistics kernel), one JSON line per shape.

    python tools/bench_mnm_vocab.py [--shapes V1,V2,V3,V4] [--sweeps 10] [--warmup 2]

Stage times come from dpmm_timing_read (CUDA events around each kernel).  Flops and bytes are computed from the
shapes here: label = 2 n K D flop against bench.py's FFMA2_PEAK_TFLOPS, and n (4 D + 4) bytes (one pass over X);
sub-label and statistics = one pass over X each, against bench.py's HBM figure.  Every X is larger than L2."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"V1": (200_000, 4096, 64), "V2": (50_000, 16384, 32), "V3": (1_000_000, 1000, 100), "V4": (1_000_000, 100, 500)}


def device_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def run_shape(pkg, tag, n, D, K, sweeps, warmup, ffma_tflops, hbm_gbs):
    import torch
    gen = torch.Generator(device="cuda").manual_seed(D + K)
    # counts with ~0.05 D words per document; generated on the device, laid out N x D (= D x N column-major)
    x = torch.poisson(torch.full((n, D), 0.05, device="cuda"), generator=gen).cpu().numpy()
    rng = np.random.default_rng(K)
    log_p = np.log(rng.dirichlet(np.ones(D), size=(K, 3))).astype(np.float32)
    w = rng.dirichlet(np.ones(K) * 5).astype(np.float32)
    lr = rng.dirichlet(np.ones(2) * 5, size=K).astype(np.float32)
    g = pkg.GpuSweep(x.T, pkg.MULTINOMIAL, seed=1)
    del x
    g.init_labels(K)
    g.set_params_multinomial(log_p, w, lr)

    def sweep():
        g.sample_labels(False)
        g.sample_sublabels()
        g.suff_stats(fetch=False)

    for _ in range(warmup):
        sweep()
    g.sync()
    g.timing_enable(True)
    g.timing_read(reset=True)
    t0 = time.perf_counter()
    for _ in range(sweeps):
        sweep()
    g.sync()
    wall = time.perf_counter() - t0
    tm = g.timing_read(reset=True)
    g.timing_enable(False)
    g.close()
    ms = {k: tm[k][0] / sweeps for k in ("label", "sort", "sublabel", "stats")}
    xbytes = n * (4.0 * D + 4)
    label_floor_ms = max(2.0 * n * K * D / (ffma_tflops * 1e12), xbytes / (hbm_gbs * 1e9)) * 1e3
    return dict(shape=tag, n=n, D=D, K=K, sweeps=sweeps,
                stage_ms=ms, sweeps_per_s=sweeps / wall,
                label_tflops=2.0 * n * K * D / (ms["label"] * 1e-3) / 1e12,
                label_frac_ffma2=2.0 * n * K * D / (ms["label"] * 1e-3) / (ffma_tflops * 1e12),
                label_frac_hbm=xbytes / (ms["label"] * 1e-3) / (hbm_gbs * 1e9),
                label_floor_ms=label_floor_ms,
                sublabel_frac_hbm=xbytes / (ms["sublabel"] * 1e-3) / (hbm_gbs * 1e9),
                stats_frac_hbm=xbytes / (ms["stats"] * 1e-3) / (hbm_gbs * 1e9))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="V1,V2,V3,V4")
    ap.add_argument("--sweeps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    import bench
    import __graft_entry__
    __graft_entry__.build()
    import dpmm_pkg
    pkg = dpmm_pkg.load()
    hbm_gbs = bench.peaks()["hbm_gbs"]
    for tag in args.shapes.split(","):
        n, D, K = SHAPES[tag]
        rec = run_shape(pkg, tag, n, D, K, args.sweeps, args.warmup, bench.FFMA2_PEAK_TFLOPS, hbm_gbs)
        name, power = device_info()
        rec.update(device=name, power_limit_and_max_sm_clock=power, ffma2_peak_tflops=bench.FFMA2_PEAK_TFLOPS,
                   hbm_gbs=hbm_gbs)
        print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
