#!/usr/bin/env python
"""bench.py -- Gibbs iterations/sec of the data-parallel sweep (BASELINE.json metric).

A "step" is one sweep of the hot path at a FROZEN converged parameter state (SURVEY.md 8d):
    [set_params] -> sample_labels -> sample_sublabels -> suff_stats (all clusters)
i.e. group_step's worker side (src/local_clusters_actions.jl:660-663) without the host's parameter
sampling.  Workload at N GPUs: BASELINE config C2 per GPU (NIW, N=1e6 points per GPU, D=32,
K_true=20, generate_gaussian_data restated), one NCCL all-reduce of the packed statistics per step.

  value  : device-timed (CUDA events) sweeps/s with X and the parameters resident in HBM
  e2e    : a COMPLETE Gibbs iteration at frozen K through the C ABI -- parameter step (posterior draws of the
           3K distributions and the weights, on the device for NIW), the sweep, the posterior step, and the
           device->host copy of what the host's Hastings moves read (counts, log marginal likelihoods, merge table);
           `e2e_host_params` is round 1's definition (host parameters H2D, sweep, statistics D2H)
  --impl reference : the restated reference (NumPy/OpenBLAS oracle) on the host cores, bounded sample
  --scaling weak (default): C2 per GPU; strong: the N=1e6 problem split over the GPUs
  --state overlap: the same shape with MixtureVar = 1 (clusters overlap: the exact-candidate path of the label
           kernel works for its living)
Unit at every N: "iters/s" = Gibbs sweeps over ONE C2-sized (1e6-point) problem per second; a weak-scaling step
over N GPUs completes N of them (config.n_points_total says how many points one step covers).
  --dump-outputs DIR: after the timed steps, writes what the last timed step computed (see dump_outputs) as
           DIR/<name>.npy, so that two builds run with the same arguments can be compared output for output
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (prior, N per GPU, D, K_true)
    "c1": ("niw", 10_000, 2, 6),
    "c2": ("niw", 1_000_000, 32, 20),
    "c3": ("mnm", 1_000_000, 100, 20),
    "c4": ("niw", 10_000_000, 5, 50),
    "c5s": ("niw", 2_000_000, 64, 100),   # a 1/50 slice of C5 (N=1e8) per GPU
    "c5": ("niw", 12_500_000, 64, 100),   # C5 itself at 8 GPUs: N = 1e8 over 8 shards (3.2 GB of X per GPU)
}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def build_case(name, rank=0, seed=0, mixture_var=100.0, shard=None):
    """Synthetic data of the named config + a frozen, converged parameter state: posterior draws of
    every cluster / sub-cluster given the ground-truth assignment (random halves as sub-clusters).
    shard = (rank, world) cuts the rank-0 data set into contiguous blocks (strong scaling)."""
    import dpmm_pkg
    pkg = dpmm_pkg.load()
    from dpmmsubclusters_jl_b200 import priors as P
    from dpmmsubclusters_jl_b200.data_generators import (generate_gaussian_data, generate_gaussian_mixture,
                                                         generate_mnmm_data)
    prior, n, D, K = WORKLOADS[name]
    alpha = 10.0
    prng = np.random.default_rng(seed + 7)            # parameter draws: identical on every rank
    if prior == "niw":
        mix = generate_gaussian_mixture(D, K, mixture_var, np.random.default_rng(seed))
        if shard is not None:
            rank = 0
        x, z, _, _ = generate_gaussian_data(n, D, K, mixture_var, np.random.default_rng(seed + 1000 + rank), mixture=mix)
        z = z.astype(np.int64)
        hyper = P.niw_hyperparams(1.0, np.zeros(D), D + 3, np.eye(D))    # fit() default, dp-parallel-sampling.jl:272-274
        # parameters come from rank 0's shard so that every rank holds the same state (for shards beyond 2e6 x 64
        # values: from a 2e6-point sample of the same mixture, generated identically on every rank)
        if n * D > 150_000_000:
            x0, z0, _, _ = generate_gaussian_data(2_000_000, D, K, mixture_var, np.random.default_rng(seed + 999), mixture=mix)
            z0 = z0.astype(np.int64)
        elif rank != 0:
            x0, z0, _, _ = generate_gaussian_data(n, D, K, mixture_var, np.random.default_rng(seed + 1000), mixture=mix)
            z0 = z0.astype(np.int64)
        else:
            x0, z0 = x, z
    else:
        x, z, _ = generate_mnmm_data(n, D, K, 50, np.random.default_rng(seed))
        hyper = P.multinomial_hyper(np.ones(D, np.float32))
        x0, z0 = x, z
    keep = [k for k in range(1, K + 1) if (z0 == k).sum() >= 2]
    Ke = len(keep)
    srng = np.random.default_rng(seed + 99)
    sub0 = srng.integers(1, 3, x0.shape[1])
    dists, counts, lrw = [], [], []
    for k in keep:
        m = z0 == k
        trip = []
        for sel in (m, m & (sub0 == 1), m & (sub0 == 2)):
            pts = x0[:, sel].astype(np.float64)
            if prior == "niw":
                ss = P.make_suff_stats(hyper, pts.shape[1], pts.sum(1), pts @ pts.T)
            else:
                ss = P.make_suff_stats(hyper, pts.shape[1], pts.sum(1))
            trip.append(P.sample_distribution(P.calc_posterior(hyper, ss), prng))
        dists.append(trip)
        counts.append(m.sum())
        lrw.append(prng.dirichlet([(m & (sub0 == 1)).sum() + alpha / 2, (m & (sub0 == 2)).sum() + alpha / 2]))
    w = prng.dirichlet(np.array(counts + [alpha], np.float64))[:-1].astype(np.float32)
    goff = 0
    if shard is not None:                      # contiguous block of the one data set (DistributedArrays layout)
        r, wsz = shard
        lo, hi = (n * r) // wsz, (n * (r + 1)) // wsz
        x, z, goff = x[:, lo:hi], z[lo:hi], lo
    # column-major D x N, the layout Julia hands over (each point contiguous): no transposition at upload
    case = dict(K=Ke, D=D, n=x.shape[1], x=np.asfortranarray(x), weights=w, lr_weights=np.asarray(lrw, np.float32),
                gt=z, name=name, goff=goff, hyper=hyper, alpha=alpha)
    if prior == "niw":
        case["kind"] = pkg.NIW
        case["mu"] = np.array([[d.μ for d in t] for t in dists], np.float32)
        case["inv_sigma"] = np.array([[d.invΣ for d in t] for t in dists], np.float32)
        case["logdet"] = np.array([[d.logdetΣ for d in t] for t in dists], np.float32)
    else:
        case["kind"] = pkg.MULTINOMIAL
        case["log_p"] = np.array([[d.α for d in t] for t in dists], np.float32)
    return case


def set_params(sw, case):
    if "mu" in case:
        sw.set_params_niw(case["mu"], case["inv_sigma"], case["logdet"], case["weights"], case["lr_weights"])
    else:
        sw.set_params_multinomial(case["log_p"], case["weights"], case["lr_weights"])


def algorithmic_work(case):
    """SURVEY.md 8d / BASELINE.md 3 per-unit figures x the units one launch processes."""
    n, D, K = case["n"], case["D"], case["K"]
    niw = "mu" in case
    w = {}
    if niw:
        w["label_flops"] = n * K * (2 * D * D + 3 * D)           # every point x K clusters: matvec 2D^2, subtract+dot 3D
        w["sublabel_flops"] = n * 2 * (2 * D * D + 3 * D)
        w["stats_bytes"] = n * (4 * D + 5) + 2 * K * (1 + D + D * D) * 8
    else:
        w["label_flops"] = n * K * 2 * D
        w["sublabel_flops"] = n * 2 * 2 * D
        w["stats_bytes"] = n * (4 * D + 5) + 2 * K * (1 + D) * 8
    w["label_bytes"] = n * (4 * D + 4)                           # read X once, write int32 label
    w["sublabel_bytes"] = n * (4 * D + 4 + 4 + 1 + 4)            # gather X, perm, label, sub-label, perm2
    return w


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained"),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self.nv, self.err = None, str(e)

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                 getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                 getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                 getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.005)

    def result(self):
        self.stop_flag = True
        self.join(timeout=2)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.sm)}


def run_reference(args):
    """`--impl reference`: the restated reference on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from oracle import cpu_sweep
    case = build_case(args.workload, 0, args.seed, mixture_var=state_var(args))
    cores = os.cpu_count() or 1
    workers = args.cpu_workers or cores
    r = cpu_sweep.time_cpu_sweep(case["x"], case, workers, steps=max(args.steps, 1), warmup=max(args.warmup, 1),
                                 target_step_s=args.cpu_step_s)
    # one step of this arm's workload covers n_total points (weak: N shards of the config, strong: the config);
    # the CPU time is extrapolated linearly from the sample; the unit counts 1e6-point (config-sized) problems
    n_total = case["n"] * (world if args.scaling == "weak" else 1)
    units = n_total / case["n"]
    ms_step = float(np.mean(r["step_s"])) * 1e3 * (n_total / r["n_sample"])
    val = units * 1e3 / ms_step
    unit = "iters/s"
    line = {"impl": "reference", "metric": "gibbs_iters_per_sec", "value": val, "unit": unit, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(case, args, world),
            "cpu_baseline": {"value": val, "unit": unit, "cores": r["workers"], "kind": "port",
                             "sample": f"{r['n_sample']} of {n_total} points (strided), {args.steps} sweeps of "
                                       f"{float(np.mean(r['step_s'])) * 1e3:.0f} ms, scaled linearly to N={n_total}; restated reference "
                                       f"(NumPy/OpenBLAS oracle), {r['workers']} worker processes x 1 BLAS thread; "
                                       f"Julia is not installed"},
            "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def state_var(args):
    return 1.0 if args.state == "overlap" else 100.0


def workload_config(case, args, world):
    prior, n, D, K = WORKLOADS[case["name"]]
    strong = args.scaling == "strong" and world > 1
    n_gpu = case["n"]
    n_total = n if strong else n * world
    return {"workload": f"{case['name'].upper()}: {'NIW Gaussian' if prior == 'niw' else 'multinomial'} N={n} points"
                        f"{' in total, split over the GPUs' if strong else ' per GPU'}, "
                        f"D={D}, K_true={K} (K={case['K']} non-empty), alpha=10, frozen K, "
                        f"{'overlapping clusters (MixtureVar=1)' if args.state == 'overlap' else 'converged state (MixtureVar=100)'}; "
                        f"step = sample_labels + sample_sublabels + suff_stats(all)",
            "n_points_per_gpu": n_gpu, "n_points_total": n_total, "D": D, "K": case["K"], "state": args.state,
            "unit_definition": f"iters/s counts Gibbs sweeps over one {n}-point problem; one step covers n_points_total points",
            "generator": f"generate_gaussian_data(N,D,K,{state_var(args):g}) restated" if prior == "niw" else "generate_mnmm_data(N,D,K,50) restated",
            "sampler": "inverse-CDF (reference semantics)",
            "parallelism": (f"points sharded over {world} GPU(s), 1 NCCL all-reduce/step" if world > 1 else "1 GPU"),
            "l2": f"inputs per step ({n_gpu * D * 4 / 1e6:.0f} MB X + labels) exceed the 126 MB L2; no explicit flush"
                  if n_gpu * D * 4 > 126e6 else "inputs fit in L2: a 256 MB buffer is written between steps of the roofline pass"}


FFMA2_PEAK_TFLOPS = 70.0   # packed FP32 FMA pipe, measured on the pool's B200 (tools/micro/ffma_bench.cu: 63-74)


def check_allreduce(pkg, g, case, args, rank, world, dist, torch):
    """Multi-GPU only, untimed: the all-reduced statistics of one sweep (every rank holds them) against the same
    sweep of the UN-SHARDED points on rank 0's GPU alone (aggregate_suff_stats, niw.jl:64-66)."""
    set_params(g, case)
    g.sample_labels(False)
    g.sample_sublabels()
    got = g.suff_stats()
    res = None
    if rank == 0:
        if args.scaling == "strong":
            full = build_case(args.workload, 0, args.seed, mixture_var=state_var(args))["x"]
        else:
            full = np.concatenate([build_case(args.workload, r, args.seed, mixture_var=state_var(args))["x"] for r in range(world)], axis=1)
        one = pkg.GpuSweep(np.asfortranarray(full), case["kind"], seed=args.seed + 1, global_offset=0, device=int(os.environ.get("LOCAL_RANK", "0")))
        set_params(one, case)
        one.sample_labels(False)
        one.sample_sublabels()
        want = one.suff_stats()
        one.close()
        counts_equal = bool(np.array_equal(got[0], want[0]))
        err = 0.0
        if got[2] is not None:
            diag = np.sqrt(np.maximum(np.einsum("msii->msi", want[2]), 1e-300))
            err = float(np.max(np.abs(got[2] - want[2]) / np.maximum(diag[..., :, None] * diag[..., None, :], 1e-30)))
            ex = float(np.max(np.abs(got[1] - want[1]) / np.maximum(np.sqrt(np.maximum(want[0], 1))[..., None] * diag, 1e-30)))
            err = max(err, ex)
        else:
            err = float(np.max(np.abs(got[1] - want[1])))
        res = {"ranks": world, "points": int(full.shape[1]), "counts_equal": counts_equal, "max_scaled_err": err,
               "what": "all-reduced statistics of one sweep vs the un-sharded sweep on one GPU (untimed)"}
        assert counts_equal and err <= 1e-4, f"all-reduced statistics differ from the un-sharded run: {res}"
    if world > 1:
        dist.barrier()
    return res


DUMP_MAX_POINTS = 1 << 21   # per-point arrays: 2 x 8 MB as float32; the statistics add at most ~10 MB (C5: K=100, D=64)


def dump_outputs(g, out_dir, write):
    """The arrays a caller of the timed sweep receives, from its last step: labels and sub-labels of this rank's
    points (float32, exact for these small integers) and the statistics of every cluster and sub-cluster (float64:
    counts, sum x, and sum x x' for NIW).  Beyond DUMP_MAX_POINTS points the labels are those of a fixed sample of
    points (the same sorted indices for every build: the sample depends only on n).  Every rank fetches (the fetch
    of the statistics is a collective); `write` says whether this one writes."""
    lab, sub = g.get_labels(), g.get_sublabels()
    counts, sum_x, sum_xx = g.suff_stats()
    if not write:
        return
    if g.n > DUMP_MAX_POINTS:
        sel = np.sort(np.random.default_rng(0).choice(g.n, DUMP_MAX_POINTS, replace=False))
        lab, sub = lab[sel], sub[sel]
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"labels": lab.astype(np.float32), "sublabels": sub.astype(np.float32),
              "counts": counts.astype(np.float64), "sum_x": sum_x}
    if sum_xx is not None:
        arrays["sum_xx"] = sum_xx
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"[bench] wrote {', '.join(arrays)} to {out_dir} ({sum(a.nbytes for a in arrays.values()) / 1e6:.1f} MB)")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed sweeps (>= 1)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--state", default="converged", choices=["converged", "overlap"])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--cpu-workers", type=int, default=0)
    ap.add_argument("--cpu-step-s", type=float, default=1.5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fit", action="store_true")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the labels, sub-labels and statistics of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import dpmm_pkg
    import __graft_entry__ as ge
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if rank == 0:
        ge.build()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: this framework has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()
    pkg = dpmm_pkg.load()
    args.warmup = max(args.warmup, 3)
    strong = args.scaling == "strong" and world > 1

    case = build_case(args.workload, rank, args.seed, mixture_var=state_var(args), shard=(rank, world) if strong else None)
    niw = "mu" in case
    t0 = time.perf_counter()
    goff = case["goff"] if strong else rank * case["n"]
    g = pkg.GpuSweep(case["x"], case["kind"], seed=args.seed + 1, global_offset=goff, device=local)
    g.sync()
    x_upload_ms = (time.perf_counter() - t0) * 1e3
    stream = torch.cuda.current_stream()
    g.set_stream(stream.cuda_stream)
    if world > 1:
        ids = [pkg.GpuSweep.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        g.comm_init(ids[0], rank, world)
    check = None
    if world > 1 and not args.no_check:
        check = check_allreduce(pkg, g, case, args, rank, world, dist, torch)
    set_params(g, case)
    sampler = ClockSampler(local)            # (NVML initialisation happens here, well before the timed region)
    warm = torch.zeros(1, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def align():
        """Ranks leave the host barrier milliseconds apart; one small all-reduce on the timing stream makes the
        timed region start together ON THE DEVICE (the first collective of the loop would absorb the skew otherwise)."""
        if world > 1:
            dist.all_reduce(warm)

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def gather_ranks(v):
        if world == 1:
            return [v]
        t = torch.zeros(world, dtype=torch.float64, device="cuda")
        t[rank] = v
        dist.all_reduce(t)
        return [float(a) for a in t.tolist()]

    def sweep_device():
        g.sample_labels(False)
        g.sample_sublabels()
        g.suff_stats(fetch=False)

    e2e_out = [None]

    def sweep_e2e_host_params():
        set_params(g, case)
        g.sample_labels(False)
        g.sample_sublabels()
        e2e_out[0] = g.suff_stats(out=e2e_out[0])   # host result arrays reused across steps, as a sampler loop would
        return e2e_out[0]

    splittable = np.ones(case["K"], bool)

    def iteration_e2e():
        """A whole Gibbs iteration at frozen K: parameter step, sweep, posterior step, scalars to the host."""
        g.sample_params(case["K"])
        g.sample_labels(False)
        g.sample_sublabels()
        return g.posterior_step(None, splittable=splittable)

    # ---- value: device-resident sweep, CUDA events on the launching stream ----
    for _ in range(args.warmup):
        sweep_device()
    # settle: the NIW label path adapts from the previous call's counters (cold labels send the next 8 calls to the
    # FMA kernel); 12 synchronised steps put the timed region in the steady state whatever the warm-up count was
    for _ in range(12):
        sweep_device()
        g.sync()
    barrier()
    sampler.start()
    l0 = g.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    align()
    e0.record(stream)
    for _ in range(args.steps):
        sweep_device()
    e1.record(stream)
    barrier()
    launches = g.launch_count() - l0
    dev_ms_rank = e0.elapsed_time(e1)
    dev_ms_all = gather_ranks(dev_ms_rank)
    dev_ms = max(dev_ms_all)
    clocks = sampler.result()
    ms_step = dev_ms / args.steps
    if args.dump_outputs:
        dump_outputs(g, args.dump_outputs, rank == 0)

    # ---- e2e (round 1's definition): host parameters in, host statistics out, every step ----
    for _ in range(3):
        sweep_e2e_host_params()
    barrier()
    align()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = sweep_e2e_host_params()
    barrier()
    e2e_hp_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / args.steps
    K, D = case["K"], case["D"]
    if niw:
        h2d_hp = 4 * (3 * K * (D + D * D + 1) + 3 * K)
        d2h_hp = 8 * 3 * K * (1 + D + D * D)
    else:
        h2d_hp = 4 * (3 * K * D + 3 * K)
        d2h_hp = 8 * 3 * K * (1 + D)
    n_total = case["n"] * world if not strong else WORKLOADS[case["name"]][1]
    assert int(out[0][:, 0].sum()) == n_total, "statistics do not cover every point"

    # ---- e2e (headline): the complete iteration with the parameter step on the device ----
    e2e_ms, h2d, d2h, e2e_what = e2e_hp_ms, h2d_hp, d2h_hp, "host parameters H2D + sweep + statistics D2H (no device parameter step for this prior)"
    if niw:
        hy = case["hyper"]
        g.set_hyper_niw(hy.κ, hy.m, hy.ν, hy.ψ, case["alpha"])
        g.posterior_step(None)         # the statistics / posterior tables of the current (converged) labels
        for _ in range(5):
            res = iteration_e2e()
        assert (res[0][:, 0] > 0).sum() == case["K"], "the e2e state lost clusters"

        barrier()
        align()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            res = iteration_e2e()
        barrier()
        e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / args.steps
        assert int(res[0][:, 0].sum()) == n_total, "statistics do not cover every point"
        h2d, d2h = K, 8 * (6 * K + K * K)
        e2e_what = ("complete Gibbs iteration at frozen K: device parameter step (3K posterior draws, weights), sweep, posterior "
                    "step (statistics, all-reduce, posteriors, log marginal likelihoods, K x K merge table), scalars D2H")
        set_params(g, case)            # back to the frozen state for the per-kernel pass

    # ---- per-kernel durations (CUDA events around every launch) for the roofline ----
    os.environ["DPMM_TC_STATS"] = "1"   # diagnostics of the tensor-core label path (which path ran, refinements/point)
    for _ in range(3):
        sweep_device()
    flush = None
    if case["n"] * D * 4 <= 126e6:
        flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    g.timing_enable(True)
    nprof = min(args.steps, 50)
    for _ in range(nprof):
        if flush is not None:
            flush.fill_(1)
        sweep_device()
    tim = g.timing_read()
    g.timing_enable(False)
    tc_pts, tc_cand, tc_ovf = g.tc_stats(overflow=True)
    os.environ.pop("DPMM_TC_STATS", None)
    work = algorithmic_work(case)
    pk = peaks()
    tf32_peak = pk["bf16_tflops"] / 2.0
    stages = {}
    for name, (ms, cnt) in tim.items():
        if cnt:
            stages[name] = {"us_per_step": ms / nprof * 1e3, "launches_per_step": cnt / nprof}
    lab_s = stages["label"]["us_per_step"] * 1e-6
    on_tc = niw and tc_pts > 0
    t2 = on_tc and D in (32, 64)
    if niw:
        name = ("gauss_label_tc2_kernel (tcgen05 kind::tf32: pivot factor + 8-row screen of every cluster on pivot-sorted, "
                "centred tiles; exact FP32 candidates; label draw)" if t2 else
                "gauss_label_warp_kernel (fused FP32 log-likelihood + label draw, packed FFMA2)")
        peak = tf32_peak if t2 else FFMA2_PEAK_TFLOPS
        issued = case["n"] * (2 * D * D + 2 * 8 * case["K"] * (D if K <= 60 and D == 32 else 8)) if t2 else work["label_flops"] / 2
        stages["label"].update({"kernel": name, "bound": "tensor" if t2 else "fma",
                                "algorithmic_tflops": work["label_flops"] / lab_s / 1e12,
                                "frac": work["label_flops"] / lab_s / 1e12 / peak, "peak_tflops": peak,
                                "issued_tflops": issued / lab_s / 1e12,
                                "hbm_gbs": work["label_bytes"] / lab_s / 1e9,
                                "hbm_frac": work["label_bytes"] / lab_s / 1e9 / pk["hbm_gbs"],
                                "exact_evaluations_per_point": (tc_cand / tc_pts) if on_tc else None,
                                "overflow_points": tc_ovf if on_tc else None})
    else:
        mtc = D % 4 == 0 and D <= 128 and K <= 32
        stages["label"].update({"kernel": "mnm_label_tc_kernel (exact 3-way TF32 split GEMM on tcgen05 + label draw)" if mtc
                                else "mnm_label_kernel (FP32 FMA pipe)", "bound": "hbm",
                                "achieved_gbs": work["label_bytes"] / lab_s / 1e9,
                                "frac": work["label_bytes"] / lab_s / 1e9 / pk["hbm_gbs"],
                                "algorithmic_tflops": work["label_flops"] / lab_s / 1e12})
    sl_s = stages["sublabel"]["us_per_step"] * 1e-6
    if "stats" in stages:
        st_s = stages["stats"]["us_per_step"] * 1e-6
        stages["stats"].update({"bound": "hbm", "achieved_gbs": work["stats_bytes"] / st_s / 1e9,
                                "frac": work["stats_bytes"] / st_s / 1e9 / pk["hbm_gbs"]})
        stages["sublabel"].update({"bound": "hbm", "achieved_gbs": work["sublabel_bytes"] / sl_s / 1e9,
                                   "frac": work["sublabel_bytes"] / sl_s / 1e9 / pk["hbm_gbs"],
                                   "algorithmic_tflops": work["sublabel_flops"] / sl_s / 1e12})
        if niw and D == 64:
            stages["stats"]["kernel"] = ("niw_stats_tc64_kernel (left / right sum x x' as tcgen05 kind::tf32 rank-8 updates, "
                                         "M = 128 x N = 64, MN-major operands; Float64 accumulators)")
            stages["sublabel"]["kernel"] = ("niw_sublabel_tc64_kernel (3-term TF32 product on tcgen05, M = N = 128, + sub-label draw) "
                                            "followed by the left / right partition pass")
    else:
        # NIW D=32: niw_substats_tc_kernel draws the sub-labels AND accumulates the statistics in ONE pass over X.
        # frac = the bytes of that one pass (B_3 of SURVEY 8d) over its time; two_stage_frac credits the bytes the two
        # separate stages would move (B_1 + B_3).
        both = work["sublabel_bytes"] + work["stats_bytes"]
        stages["sublabel"].update({"kernel": "niw_substats_tc_kernel (sub-label draw + left/right statistics, fused, tcgen05)",
                                   "fused_stages": ["sublabel", "stats"], "bound": "hbm",
                                   "achieved_gbs": work["stats_bytes"] / sl_s / 1e9,
                                   "frac": work["stats_bytes"] / sl_s / 1e9 / pk["hbm_gbs"],
                                   "two_stage_gbs": both / sl_s / 1e9, "two_stage_frac": both / sl_s / 1e9 / pk["hbm_gbs"],
                                   "algorithmic_tflops": work["sublabel_flops"] / sl_s / 1e12})
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    tj = json.load(open(tp)) if os.path.exists(tp) else {}
    # the dominant kernel of the step by measured time
    dom = max((k for k in ("label", "sublabel", "stats") if k in stages), key=lambda k: stages[k]["us_per_step"])
    ds = stages[dom]
    traffic = tj.get(case["name"], {}).get({"label": "label_tc2", "sublabel": "sublabel_stats_fused" if "fused_stages" in ds else "sublabel",
                                            "stats": "stats"}[dom])
    if ds["bound"] == "hbm":
        roofline = {"kernel": ds.get("kernel", dom), "stage": dom, "bound": "hbm", "achieved": ds["achieved_gbs"], "peak": pk["hbm_gbs"],
                    "unit": "GB/s", "frac": ds["frac"], "traffic": traffic, "peak_source": pk["source"],
                    "algorithmic_bytes_per_launch": work["stats_bytes"] if dom != "label" else work["label_bytes"]}
        if "fused_stages" in ds:
            roofline["note"] = ("HBM is the roofline this pass is measured against by its bytes; what bounds the kernel is the shared-memory "
                                "data pipe: ncu l1tex__data_pipe_lsu_wavefronts 55 % + l1tex__data_pipe_tc_wavefronts_mem_shared 35 % of "
                                "peak, DRAM 20 %, tensor pipe 27 % (profiles/r2n_ncu_summary.md, DESIGN.md section 4)")
    else:
        roofline = {"kernel": ds["kernel"], "stage": dom, "bound": "tensor" if ds["bound"] == "tensor" else "tensor",
                    "achieved": ds["algorithmic_tflops"], "peak": ds["peak_tflops"], "unit": "TFLOP/s", "frac": ds["frac"],
                    "traffic": traffic,
                    "peak_source": (f"TF32 dense = 1/2 x bf16 {pk['bf16_tflops']} TFLOP/s, {pk['source']}" if ds["bound"] == "tensor"
                                    else "packed FP32 FFMA2 pipe, measured with tools/micro/ffma_bench.cu on this pool's B200 (the FMA pipe, not the tensor pipe, bounds this shape: D < 32)"),
                    "algorithmic_flops_per_launch": work["label_flops"], "issued_tflops": ds.get("issued_tflops"),
                    "note": "achieved = ALGORITHMIC flops (N K (2 D^2 + 3 D), SURVEY 8d) / time; the screen issues fewer (issued_tflops)"}

    line = None
    if rank == 0:
        units = 1.0 if strong else float(world)
        line = {"metric": "gibbs_iters_per_sec", "value": units * 1e3 / ms_step, "unit": "iters/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": workload_config(case, args, world),
                "job_iters_per_s": 1e3 / ms_step,
                "e2e": {"value": units * 1e3 / e2e_ms, "unit": "iters/s", "ms_per_step": e2e_ms,
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "what": e2e_what,
                        "note": "X stays resident across iterations as in fit(); its one-time upload is x_upload_ms"},
                "e2e_host_params": {"value": units * 1e3 / e2e_hp_ms, "unit": "iters/s", "ms_per_step": e2e_hp_ms,
                                    "h2d_bytes_per_step": h2d_hp, "d2h_bytes_per_step": d2h_hp,
                                    "what": "host parameters H2D + pack + sweep + statistics D2H (no parameter sampling)"},
                "x_upload_ms": x_upload_ms, "x_bytes": int(case["n"] * D * 4),
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "stages": stages,
                "rank_ms_per_step": [m / args.steps for m in dev_ms_all],
                "rank_skew_ms_per_step": (max(dev_ms_all) - min(dev_ms_all)) / args.steps}
        if check is not None:
            line["allreduce_check"] = check
    g.close()
    # ---- CPU baseline beside it (rank 0, N=1 only) ----
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import cpu_sweep
        cores = os.cpu_count() or 1
        workers = args.cpu_workers or cores
        r = cpu_sweep.time_cpu_sweep(case["x"], case, workers, steps=4, warmup=1, target_step_s=args.cpu_step_s)
        scale = case["n"] / r["n_sample"]
        cpu_ms = float(np.mean(r["step_s"])) * 1e3 * scale
        line["cpu_baseline"] = {"value": 1e3 / cpu_ms, "unit": "iters/s", "cores": r["workers"], "kind": "port",
                                "sample": f"{r['n_sample']} of {case['n']} points (strided), 4 sweeps, scaled linearly; "
                                          f"restated reference (NumPy/OpenBLAS oracle), {r['workers']} worker processes "
                                          f"x 1 BLAS thread, host has {cores} cores; Julia is not installed"}
    # ---- a complete fit() on the same data (parameter step on the device for NIW): NMI, final K ----
    if rank == 0 and world == 1 and not args.no_fit:
        from dpmmsubclusters_jl_b200.host import normalized_mutual_info
        fits = []
        for rep in range(2):           # the first call also pays CUDA module loading and the kernels' first launches
            t0 = time.perf_counter()
            if niw:
                out = pkg.fit(case["x"], 10.0, iters=100, seed=args.seed + 1, burnout=20)
            else:
                out = pkg.fit(case["x"], pkg.multinomial_hyper(np.ones(case["D"], np.float32)), 10.0, iters=100,
                              seed=args.seed + 1, burnout=20)
            fits.append((time.perf_counter() - t0, out))
        dt, out = fits[-1]
        line["fit"] = {"iters": 100, "seconds": dt, "iters_per_s": 100 / dt, "loop_seconds": float(sum(out[3])),
                       "loop_iters_per_s": 100 / float(sum(out[3])), "first_call_seconds": fits[0][0],
                       "final_K": len(out[1]), "K_true_nonempty": int(len(np.unique(case["gt"]))),
                       "nmi": normalized_mutual_info(case["gt"], out[0]),
                       "note": "fit(x, alpha=10, iters=100, burnout=20) from K=1, second call in the process. iters_per_s: the "
                               "whole call (X upload, 100 Gibbs iterations with split/merge moves, label download, result "
                               "objects); loop_iters_per_s: sum of the per-iteration times fit() itself reports (iter_count, "
                               "dp-parallel-sampling.jl:389-390). Parameter step: " + ("device" if niw else "host (NumPy)")}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
