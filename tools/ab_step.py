#!/usr/bin/env python
"""Interleaved A/B timing of whole benchmark steps in ONE process on ONE model (cfg3 by default).

    python tools/ab_step.py "mb=512,retain=auto" "mb=768,retain=auto" "mb=512,retain=auto,accum=0" ...

Boxes differ by several percent in sustained clocks under the power cap, and one box drifts while it
warms up, so configurations are compared round-robin (A B C A B C ...) inside one process: `rounds`
passes over the list, each entry 1 untimed + `steps` timed steps, CUDA events.  Keys: mb (micro-batch),
retain ("auto" | int), accum (0/1: in-place gradient accumulation of the non-final chunks), alloc
("expandable": torch allocator expandable segments - must be the same for every entry, applied at start).
Diagnostic tool - never a bench value."""
from __future__ import annotations

import json
import os
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def parse(spec):
    d = dict(mb=512, retain="auto", accum=1)
    for kv in filter(None, spec.split(",")):
        k, v = kv.split("=")
        d[k] = v
    d["mb"] = int(d["mb"])
    d["accum"] = int(d["accum"])
    d["retain"] = d["retain"] if d["retain"] == "auto" else int(d["retain"])
    return d


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    opts = dict(a[2:].split("=") for a in sys.argv[1:] if a.startswith("--"))
    rounds, steps = int(opts.get("rounds", 2)), int(opts.get("steps", 3))
    batch = int(opts.get("batch", 4096))
    workload = opts.get("workload", "cfg3")
    if opts.get("alloc") == "expandable":
        os.environ["PYTORCH_CUDA_ALLOC_CONF"] = "expandable_segments:True"
    import torch
    import bench
    from x_clip_b200 import engine
    cfgs = [parse(a) for a in args] or [parse("")]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    run = bench.Runner(bench.WORKLOADS[workload][0], "nce", batch, cfgs[0]["mb"], 0.5, dev, 0, 1,
                       retain=cfgs[0]["retain"])
    results = [[] for _ in cfgs]
    for r in range(rounds):
        for i, c in enumerate(cfgs):
            run.clip.microbatch = c["mb"]
            run.clip.microbatch_retain = c["retain"]
            engine.INPLACE_GRAD_ACCUMULATION = bool(c["accum"])
            run.step()
            torch.cuda.synchronize()
            s0 = torch.cuda.memory_stats(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                loss = run.step()
            e1.record()
            torch.cuda.synchronize()
            s1 = torch.cuda.memory_stats(dev)
            ms = e0.elapsed_time(e1) / steps
            results[i].append(ms)
            print(json.dumps({"round": r, "cfg": args[i] if args else "", "ms_per_step": round(ms, 2),
                              "pairs_per_s": round(batch / ms * 1e3, 1), "loss": round(loss.item(), 4),
                              "plan": run.clip.last_step_plan,
                              "device_allocs": s1["num_device_alloc"] - s0["num_device_alloc"],
                              "device_frees": s1["num_device_free"] - s0["num_device_free"],
                              "alloc_retries": s1["num_alloc_retries"] - s0["num_alloc_retries"],
                              "peak_GB": round(torch.cuda.max_memory_allocated(dev) / 1e9, 1)}), flush=True)
            torch.cuda.reset_peak_memory_stats(dev)
    print("== summary (ms/step per round)")
    for a, rs in zip(args or [""], results):
        print(f"{a:50s} " + " ".join(f"{x:8.2f}" for x in rs) + f"   min {min(rs):8.2f}")


if __name__ == "__main__":
    main()
