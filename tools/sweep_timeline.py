"""Device timeline of the benchmarked sweep: every kernel, memset and copy that one `sweep_device()` step of
bench.py (sample_labels + sample_sublabels + suff_stats(all), no fetch) puts on the stream, with its duration
and the idle gap before it, averaged over the recorded steps.

    python tools/sweep_timeline.py [--workload c2] [--state converged] [--steps 50] [--out DIR]

The gaps are what the kernels themselves do not explain: launch latency, memset / copy nodes and the
prologue of the next kernel until its first instruction.  Kernels chained by programmatic dependent launch
start before their predecessor ends, so their rows show no gap and a duration that includes the wait for the
predecessor; the per-step span is then the figure to compare.  The profiler adds a little host overhead per
launch, so take the per-step total from bench.py and the split from here.  --out writes the Chrome trace.
"""
import argparse
import os
import subprocess
import sys
from collections import defaultdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q or "unknown"
    except Exception as e:  # pragma: no cover
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c2")
    ap.add_argument("--state", default="converged", choices=["converged", "overlap"])
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None, help="directory for the Chrome trace")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    import bench
    import dpmm_pkg
    import __graft_entry__ as ge
    ge.build()
    if not torch.cuda.is_available():
        raise SystemExit("sweep_timeline.py needs a CUDA device")
    pkg = dpmm_pkg.load()
    case = bench.build_case(args.workload, 0, args.seed, mixture_var=1.0 if args.state == "overlap" else 100.0)
    g = pkg.GpuSweep(case["x"], case["kind"], seed=args.seed + 1, global_offset=0, device=0)
    stream = torch.cuda.current_stream()
    g.set_stream(stream.cuda_stream)
    bench.set_params(g, case)

    def sweep_device():
        g.sample_labels(False)
        g.sample_sublabels()
        g.suff_stats(fetch=False)

    for _ in range(args.warmup):
        sweep_device()
    for _ in range(12):            # the settle of bench.py: the adaptive label path reads the previous call's counters
        sweep_device()
        g.sync()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps):
            sweep_device()
        torch.cuda.synchronize()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        prof.export_chrome_trace(os.path.join(args.out, f"sweep_timeline_{args.workload}_{args.state}.pt.trace.json"))

    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and e.time_range.elapsed_us() >= 0]
    ev.sort(key=lambda e: e.time_range.start)
    if not ev:
        raise SystemExit("the profiler recorded no device activity")
    span = ev[-1].time_range.end - ev[0].time_range.start
    rows = defaultdict(lambda: [0, 0.0, 0.0])   # name -> count, busy us, gap-before us
    order = []
    prev_end = None
    for e in ev:
        name = e.name if len(e.name) <= 60 else e.name[:57] + "..."
        r = rows[name]
        if r[0] == 0:
            order.append(name)
        r[0] += 1
        r[1] += e.time_range.elapsed_us()
        if prev_end is not None:
            r[2] += max(0.0, e.time_range.start - prev_end)
        prev_end = max(prev_end or 0, e.time_range.end)
    n = args.steps
    print(f"card: {card()}")
    print(f"workload {args.workload} ({args.state}), {n} steps recorded, {len(ev) / n:.2f} device ops per step, "
          f"{span / n:.1f} us per step (first op start to last op end / steps)")
    print(f"{'op':<62}{'per step':>9}{'us each':>10}{'gap before':>12}")
    busy = gaps = 0.0
    for name in order:
        c, t, gp = rows[name]
        busy += t
        gaps += gp
        print(f"{name:<62}{c / n:>9.2f}{t / c:>10.2f}{gp / c:>12.2f}")
    print(f"per step: busy {busy / n:.1f} us, gaps {gaps / n:.1f} us")
    g.close()


if __name__ == "__main__":
    main()
