#!/usr/bin/env python
"""Per-kernel device time of the bench.py device step, from torch.profiler (CUDA activities), in a run of its own.

The step is bench.py's: the same make_workload, one GangPacker(async_snapshot=True), set_snapshot_device +
pack_batch_device on the library's stream, captured into a CUDA graph and replayed, the L2 flushed before every step.
Prints one line per kernel (and per memset / memcpy node) with its device time per step and writes the same as JSON to
OUT_DIR/step_profile_<workload>.json.  Profiling slows the host, so step times belong to bench.py; this breakdown says
where the device time of a step goes.

    python tools/step_profile.py OUT_DIR [--workload tightly-100k] [--steps 200] [--warmup 20]
"""
import argparse
import collections
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from bench import APP_KEYS, WORKLOADS, make_workload      # noqa: E402


def gpu_facts():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else ""
    except (OSError, subprocess.SubprocessError):
        return ""


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--workload", default="tightly-100k", choices=sorted(WORKLOADS))
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    import k8s_spark_scheduler_b200 as g
    if not torch.cuda.is_available():
        raise SystemExit("step_profile.py needs a CUDA device")
    w = WORKLOADS[args.workload]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    packer = g.GangPacker(device=0, async_snapshot=True)
    stream = torch.cuda.ExternalStream(packer.stream_handle(), device=dev)
    nodes, a, eoff, eorder = make_workload(w, 0)
    q = len(a["count"])
    total_exec = int(a["off"][-1])

    def dev_t(x, dtype):
        return torch.from_numpy(np.ascontiguousarray(x)).to(dtype).to(dev)

    n_nodes, n_ord = w["nodes"], len(eorder)
    snapbuf = torch.zeros(3 * n_nodes + (n_ord + 1) // 2, dtype=torch.int64, device=dev)
    tn = {"cpu": snapbuf[0:n_nodes], "mem": snapbuf[n_nodes:2 * n_nodes], "gpu": snapbuf[2 * n_nodes:3 * n_nodes],
          "eorder": snapbuf[3 * n_nodes:].view(torch.int32)[:n_ord], "eoff": dev_t(eoff, torch.int32)}
    tn["cpu"].copy_(dev_t(nodes["avail_cpu"], torch.int64)); tn["mem"].copy_(dev_t(nodes["avail_mem"], torch.int64))
    tn["gpu"].copy_(dev_t(nodes["avail_gpu"], torch.int64)); tn["eorder"].copy_(dev_t(eorder, torch.int32))
    ta = {k: dev_t(a[k], torch.int64 if a[k].dtype == np.int64 else (torch.uint8 if a[k].dtype == np.uint8 else torch.int32))
          for k in APP_KEYS}
    ta["off"] = dev_t(a["off"], torch.int64)
    if w["groups"] == 1:
        ta.pop("group")
    if w["mode"] == 0:
        ta.pop("young")
    d_driver = torch.empty(q, dtype=torch.int32, device=dev)
    d_exec = torch.empty(max(total_exec, 1), dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    torch.cuda.synchronize()

    def device_step():
        packer.set_snapshot_device(tn["cpu"], tn["mem"], tn["gpu"], tn["eoff"], tn["eorder"], tn["eoff"], tn["eorder"])
        packer.pack_batch_device(ta, w["algo"], w["mode"], d_driver, d_exec)

    with torch.cuda.stream(stream):
        for _ in range(max(args.warmup, 3)):
            flush.fill_(1)
            device_step()
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            device_step()
        for _ in range(2):
            graph.replay()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for s in range(args.steps):
                flush.fill_(s & 0xff)
                graph.replay()
            torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    events = trace["traceEvents"] if isinstance(trace, dict) else trace
    dur = collections.defaultdict(float)
    calls = collections.Counter()
    for e in events:
        if e.get("ph") != "X" or e.get("cat") not in ("kernel", "gpu_memset", "gpu_memcpy"):
            continue
        name = e["name"]
        if "FillFunctor" in name:          # the L2 flush between steps
            continue
        dur[name] += float(e["dur"])
        calls[name] += 1
    rows = sorted(({"name": n, "us_per_step": dur[n] / args.steps, "calls_per_step": calls[n] / args.steps} for n in dur),
                  key=lambda r: -r["us_per_step"])
    step_us = sum(r["us_per_step"] for r in rows)
    res = {"workload": args.workload, "steps": args.steps, "gpu": gpu_facts(), "device_us_per_step": step_us,
           "kernels": rows, "source": "torch.profiler CUDA activities, CUDA-graph replay of the bench.py device step"}
    os.makedirs(args.out_dir, exist_ok=True)
    out = os.path.join(args.out_dir, f"step_profile_{args.workload}.json")
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(f"{args.workload}: {step_us:.1f} us of device time per step ({res['gpu']})")
    for r in rows:
        print(f"  {r['us_per_step']:8.2f} us  x{r['calls_per_step']:.0f}  {r['name'][:140]}")
    print("wrote", out)
    del graph, snapbuf, tn, ta, d_driver, d_exec, flush
    packer.close()


if __name__ == "__main__":
    main()
