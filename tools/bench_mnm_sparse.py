"""Per-stage device times of multinomial sweeps on sparse counts (dpmm_create_sparse) against the dense context holding
the same matrix, one JSON line per (shape, form), written to profiles/mnm_sparse_bench.jsonl (--out) and stdout.

    python tools/bench_mnm_sparse.py [--shapes V1,V2,V3,V4,S1] [--sweeps 10] [--warmup 2] [--out PATH]

V1-V4 are the shapes of tools/bench_mnm_vocab.py (Poisson(0.05) counts: about 5 % of the entries are non-zero); their
sparse and dense contexts live side by side and their sweeps alternate after the warm-up, so that both forms see the
same machine state.  S1 (n = 2e6, D = 16 384, about 100 words per document, 131 GB dense) runs in sparse form only.
Stage times come from dpmm_timing_read (CUDA events around each kernel).  Work is computed from the shapes here:
the dense label stage does 2 n K D flop, the sparse one 2 nnz K; the dense sub-label and statistics stages read X once
(n (4 D + 4) bytes), the sparse ones the compressed rows once (8 nnz + 8 (n + 1) bytes)."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_mnm_vocab import SHAPES, device_info  # noqa: E402

S1 = (2_000_000, 16384, 200, 100)   # n, D, K, words per document


def params(D, K):
    rng = np.random.default_rng(K)
    log_p = np.log(rng.dirichlet(np.ones(D), size=(K, 3))).astype(np.float32)
    w = rng.dirichlet(np.ones(K) * 5).astype(np.float32)
    lr = rng.dirichlet(np.ones(2) * 5, size=K).astype(np.float32)
    return log_p, w, lr


def open_sweep(pkg, x, D, K):
    g = pkg.GpuSweep(x, pkg.MULTINOMIAL, seed=1)
    g.init_labels(K)
    g.set_params_multinomial(*params(D, K))
    return g


def sweep(g):
    g.sample_labels(False)
    g.sample_sublabels()
    g.suff_stats(fetch=False)


def timed(gs, sweeps, warmup):
    """Warm every context up, then run `sweeps` sweeps of each, alternating; per-stage ms per sweep and sweeps/s."""
    for g in gs:
        for _ in range(warmup):
            sweep(g)
        g.sync()
        g.timing_enable(True)
        g.timing_read(reset=True)
    wall = [0.0] * len(gs)
    for _ in range(sweeps):
        for i, g in enumerate(gs):
            t0 = time.perf_counter()
            sweep(g)
            g.sync()
            wall[i] += time.perf_counter() - t0
    out = []
    for i, g in enumerate(gs):
        tm = g.timing_read(reset=True)
        g.timing_enable(False)
        out.append(({k: tm[k][0] / sweeps for k in ("label", "sort", "sublabel", "stats", "stats_aux")}, sweeps / wall[i]))
    return out


def record(tag, form, n, D, K, nnz, ms, rate, ffma_tflops, hbm_gbs):
    if form == "dense":
        flop, xbytes = 2.0 * n * K * D, n * (4.0 * D + 4)
    else:
        flop, xbytes = 2.0 * nnz * K, 8.0 * nnz + 8.0 * (n + 1)
    return dict(shape=tag, form=form, n=n, D=D, K=K, nnz=int(nnz), stage_ms=ms, sweeps_per_s=rate,
                label_frac_ffma2=flop / (ms["label"] * 1e-3) / (ffma_tflops * 1e12),
                sublabel_frac_hbm=xbytes / (ms["sublabel"] * 1e-3) / (hbm_gbs * 1e9),
                stats_frac_hbm=xbytes / (ms["stats"] * 1e-3) / (hbm_gbs * 1e9))


def s1_matrix(n, D, words, rng):
    """CSC [D, n] with `words` uniform draws per document (duplicates summed by the sweep's conversion)."""
    import scipy.sparse as sps
    rows = np.sort(rng.integers(0, D, (n, words), dtype=np.int32), axis=1).reshape(-1)
    indptr = np.arange(0, (n + 1) * words, words, dtype=np.int64)
    return sps.csc_matrix((np.ones(rows.size, np.float32), rows, indptr), shape=(D, n))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="V1,V2,V3,V4,S1")
    ap.add_argument("--sweeps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mnm_sparse_bench.jsonl"))
    args = ap.parse_args()
    import scipy.sparse as sps
    import torch
    import bench
    import __graft_entry__
    __graft_entry__.build()
    import dpmm_pkg
    pkg = dpmm_pkg.load()
    hbm_gbs = bench.peaks()["hbm_gbs"]
    name, power = device_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for tag in args.shapes.split(","):
            recs = []
            if tag == "S1":
                n, D, K, words = S1
                x = s1_matrix(n, D, words, np.random.default_rng(5))
                gs = [open_sweep(pkg, x, D, K)]
                nnz = int(x.nnz)
                del x
                (ms, rate), = timed(gs, args.sweeps, args.warmup)
                recs.append(record(tag, "sparse", n, D, K, nnz, ms, rate, bench.FFMA2_PEAK_TFLOPS, hbm_gbs))
            else:
                n, D, K = SHAPES[tag]
                gen = torch.Generator(device="cuda").manual_seed(D + K)
                x = torch.poisson(torch.full((n, D), 0.05, device="cuda"), generator=gen).cpu().numpy()   # N x D
                xs = sps.csr_matrix(x).T        # D x N, CSC
                nnz = int(xs.nnz)
                gs = [open_sweep(pkg, x.T, D, K), open_sweep(pkg, xs, D, K)]
                del x, xs
                res = timed(gs, args.sweeps, args.warmup)
                for form, (ms, rate) in zip(("dense", "sparse"), res):
                    recs.append(record(tag, form, n, D, K, nnz, ms, rate, bench.FFMA2_PEAK_TFLOPS, hbm_gbs))
            for g in gs:
                g.close()
            for rec in recs:
                rec.update(device=name, power_limit_and_max_sm_clock=power, ffma2_peak_tflops=bench.FFMA2_PEAK_TFLOPS,
                           hbm_gbs=hbm_gbs, sweeps=args.sweeps)
                line = json.dumps(rec)
                print(line, flush=True)
                f.write(line + "\n")
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
