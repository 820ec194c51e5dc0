"""Per-kernel device time of the flagship workload: optimize(10) on resident cfg-2 windows (592 by default, as in
bench.py), profiled with torch.profiler (CUDA activities; the library's own streams and CUDA-graph launches are
recorded too).  Prints the mean time per launch of every kernel, writes the Chrome trace and a JSON summary under
OUT_DIR.  Needs a CUDA device.

    python tools/kernel_times.py OUT_DIR [--batch 592] [--steps 3] [--warmup 2]
"""
import argparse
import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ITERS = 10


def short_name(name):
    """'void okb::k_solve<256>(okb::WinDev const*, ...)' -> 'k_solve<256>'."""
    head = name.split("(")[0].strip()
    return re.sub(r"^(void\s+)?[\w:]*::", "", head)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("out_dir")
    ap.add_argument("--batch", type=int, default=592, help="resident cfg-2 windows")
    ap.add_argument("--distinct", type=int, default=8, help="distinct synthetic windows (replicated to fill the batch)")
    ap.add_argument("--steps", type=int, default=3, help="profiled reset + optimize(10) steps")
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    from okvis_b200 import capi, synthetic
    if not torch.cuda.is_available():
        sys.exit("kernel_times.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B = args.batch
    ctx = capi.Context(0, B)
    windows = [synthetic.make_window(2, i) for i in range(args.distinct)]
    ctx.upload_batch(0, [windows[i % len(windows)] for i in range(B)], 8)

    def step():
        ctx.reset(0, B)
        return ctx.optimize(0, B, max_iterations=ITERS)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize(dev)
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps):
            step()
        torch.cuda.synchronize(dev)
    os.makedirs(args.out_dir, exist_ok=True)
    trace = os.path.join(args.out_dir, "kernel_times_trace.json")
    prof.export_chrome_trace(trace)

    stats = {}
    with open(trace) as f:
        events = json.load(f)["traceEvents"]
    for ev in events:           # every kernel on every stream, graph launches included
        if ev.get("cat") != "kernel":
            continue
        s = stats.setdefault(short_name(ev["name"]), {"launches": 0, "total_us": 0.0})
        s["launches"] += 1
        s["total_us"] += float(ev["dur"])
    for s in stats.values():
        s["mean_us"] = s["total_us"] / s["launches"]
    props = torch.cuda.get_device_properties(dev)
    summary = {"device": props.name, "batch": B, "steps": args.steps, "iterations_per_optimize": ITERS, "kernels": stats}
    with open(os.path.join(args.out_dir, "kernel_times.json"), "w") as f:
        json.dump(summary, f, indent=1)
    print("%s, %d cfg-2 windows, %d x optimize(%d)" % (props.name, B, args.steps, ITERS))
    print("%-24s %9s %12s %10s" % ("kernel", "launches", "total ms", "mean us"))
    for name, s in sorted(stats.items(), key=lambda kv: -kv[1]["total_us"]):
        print("%-24s %9d %12.3f %10.2f" % (name, s["launches"], s["total_us"] * 1e-3, s["mean_us"]))
    ctx.close()


if __name__ == "__main__":
    main()
