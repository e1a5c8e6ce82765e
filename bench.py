#!/usr/bin/env python
"""bench.py -- gang placements/sec of the B200 bin-packer on the BASELINE workload.

    python bench.py --gpus N --steps K --warmup W          (N>1: launched by torch.distributed.run)
    python bench.py --impl reference ...                   (CPU restatement of the reference path)
    python bench.py ... --dump-outputs DIR                 (also writes the placements of the last timed step)

A "step" is one pass of the hot path over one batch of synthetic input: the 10 000-node snapshot is
laid out on the device (gp_set_snapshot_device) and 100 000 pending applications are packed
(tightly-pack, independent decisions against that snapshot) by prep + pack kernels.  With N>1 every
rank packs its own 100 000 applications (weak scaling).

value : decisions/s with inputs resident in HBM (every rank: snapshot + its block of the queue), no collective
        in the data path, CUDA events on the launch stream, L2 flushed between steps (outside the per-step
        event pairs), max over ranks.
e2e   : host buffers in, host results out.  N=1: gp_set_snapshot + gp_pack_batch from pinned memory through
        the C ABI.  N>1: rank 0 uploads the snapshot, ONE NCCL broadcast distributes it, every rank packs its
        host-resident block, the placements are all-gathered over NVLink (overlapped chunk by chunk with the
        packing) and rank 0 copies all of them to host memory.  Wall clock, max over ranks.
roofline / cpu_baseline: see DESIGN.md section 6.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (nodes, apps per GPU, algo, mode, groups)
    "tightly-100k": dict(nodes=10000, apps=100000, algo=0, mode=0, groups=1,
                         desc="10k nodes x 100k pending apps, tightly-pack, independent decisions vs one snapshot "
                              "(BASELINE.json metric / north_star size; configs[1] shape)"),
    "tightly-10k": dict(nodes=10000, apps=10000, algo=0, mode=0, groups=1,
                        desc="10k nodes x 10k pending apps, tightly-pack, independent (BASELINE configs[1])"),
    "evenly-100k": dict(nodes=10000, apps=100000, algo=1, mode=0, groups=1,
                        desc="10k nodes x 100k pending apps, distribute-evenly, independent (BASELINE configs[2])"),
    "minfrag-100k": dict(nodes=10000, apps=100000, algo=2, mode=0, groups=1,
                         desc="10k nodes x 100k pending apps, minimal-fragmentation (the per-zone packer of "
                              "single-az-minimal-fragmentation), independent; every decision is several full passes over the nodes"),
    "fifo-10k": dict(nodes=10000, apps=10000, algo=0, mode=1, groups=1,
                     desc="10k nodes x 10k pending apps, tightly-pack, FIFO (reference usage accounting), 1 instance group"),
    "fifo-da-50k": dict(nodes=10000, apps=50000, algo=0, mode=1, groups=16, da=True,
                        desc="dynamic-allocation sweep, 10k nodes x 50k apps, FIFO on, 16 instance groups (BASELINE configs[3])"),
    "tightly-100k-deep": dict(nodes=10000, apps=100000, algo=0, mode=0, groups=1, fill=(0.95, 1.0), deep=True,
                              desc="10k nodes x 100k pending apps, tightly-pack, independent, DEEP scans: cluster 95-100 % full "
                                   "(97.5 % on average), gangs of 4..128 executors that walk ~8 000 nodes of the priority order, one "
                                   "third of the applications fit nowhere (full-table scan, no fit)"),
    "evenly-100k-deep": dict(nodes=10000, apps=100000, algo=1, mode=0, groups=1, fill=(0.95, 1.0), deep=True,
                             desc="same deep-scan cluster and queue, distribute-evenly"),
    "tightly-50k-1m": dict(nodes=50000, apps=125000, algo=0, mode=0, groups=1,
                           desc="50k nodes x 1M pending apps over 8 GPUs (125k per GPU), tightly-pack (BASELINE configs[4])"),
}
ALGO_NAME = {0: "tightly-pack", 1: "distribute-evenly", 2: "minimal-fragmentation"}
ORC_ALGO = {0: 0, 1: 1, 2: 4}      # gp_algo -> oracle algo id (oracle/gangpack_oracle.h)
MODE_NAME = {0: "independent", 1: "fifo-reference", 2: "fifo-exact"}
APP_KEYS = ("drv_cpu", "drv_mem", "drv_gpu", "exe_cpu", "exe_mem", "exe_gpu", "count", "group", "young")


# ------------------------------------------------------------------------------------------------
def make_workload(w: dict, rank: int):
    from k8s_spark_scheduler_b200 import synth
    nodes = synth.make_nodes(w["nodes"], groups=w["groups"], fill=w.get("fill", (0.0, 0.9)))
    # every rank gets a different slice of the (conceptually N x apps long) queue
    apps = synth.make_apps(w["apps"], seed=synth.APP_SEED + 7919 * rank, groups=w["groups"],
                           da_sweep=bool(w.get("da")), deep=bool(w.get("deep")))
    eoff, eorder = synth.group_orders(nodes)
    a = {k: apps[k] for k in APP_KEYS}
    a["off"] = synth.exec_offsets(apps["count"])
    return nodes, a, eoff, eorder


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.idx = device_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active") and not v.lower().startswith("not"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_reference_run(w: dict, sample_apps: int, threads: int, repeats: int = 1):
    """Times the literal CPU restatement of the reference path (oracle/, kind 'port') on a bounded
    sample of the same workload, with ComputePackingEfficiencies on (the reference runs it inside
    SparkBinPack on every successful pack, binpack.go:77).
    Returns (apps timed, threads used, [seconds per repeat], results) where results is a list of
    (queue indices, driver_node, executor_nodes, exec offsets) in NODE-TABLE indices -- what the parity word of
    the bench line is checked against (outside every timed region)."""
    from k8s_spark_scheduler_b200 import synth
    from oracle import oracle as orc
    nodes, a, eoff, eorder = make_workload(w, 0)
    names = synth.node_names(w["nodes"])
    q = min(sample_apps, len(a["count"]))
    drv = orc.res_array(a["drv_cpu"][:q], a["drv_mem"][:q], a["drv_gpu"][:q])
    exe = orc.res_array(a["exe_cpu"][:q], a["exe_mem"][:q], a["exe_gpu"][:q])
    count = a["count"][:q]
    times, results = [], []
    if w["groups"] == 1:
        onames = [names[i] for i in eorder]
        for _ in range(repeats):
            cl = orc.Cluster(names, nodes["avail_cpu"], nodes["avail_mem"], nodes["avail_gpu"],
                             sched=(nodes["alloc_cpu"], nodes["alloc_mem"], nodes["alloc_gpu"]))
            t0 = time.perf_counter()
            if w["mode"] == 0:
                dn, en, off = cl.binpack_batch(ORC_ALGO[w["algo"]], drv, exe, count, onames, onames, with_efficiencies=True, n_threads=threads)
            else:
                _, dn, en, off = cl.fifo(ORC_ALGO[w["algo"]], w["mode"], drv, exe, count, a["young"][:q], onames, onames, with_efficiencies=True)
            times.append(time.perf_counter() - t0)
            results = [(np.arange(q), dn, en, off)]
        used_threads = threads if w["mode"] == 0 else 1
    else:
        # FIFO per instance group: groups are independent queues -> one thread per group
        import concurrent.futures as cf
        def run_group(g):
            sel = np.nonzero(a["group"][:q] == g)[0]
            order = eorder[eoff[g]:eoff[g + 1]]
            sub_names = [names[i] for i in order]
            cl = orc.Cluster(sub_names, nodes["avail_cpu"][order], nodes["avail_mem"][order], nodes["avail_gpu"][order],
                             sched=(nodes["alloc_cpu"][order], nodes["alloc_mem"][order], nodes["alloc_gpu"][order]))
            if w["mode"] == 0:
                dn, en, off = cl.binpack_batch(ORC_ALGO[w["algo"]], drv[sel], exe[sel], count[sel], sub_names, sub_names, True, 1)
            else:
                _, dn, en, off = cl.fifo(ORC_ALGO[w["algo"]], w["mode"], drv[sel], exe[sel], count[sel], a["young"][:q][sel], sub_names, sub_names, True)
            # sub-cluster indices -> node-table indices
            return sel, np.where(dn >= 0, order[np.maximum(dn, 0)], dn), order[np.maximum(en, 0)], off
        used_threads = min(threads, w["groups"])
        for _ in range(repeats):
            t0 = time.perf_counter()
            with cf.ThreadPoolExecutor(used_threads) as ex:   # ctypes releases the GIL
                results = list(ex.map(run_group, range(w["groups"])))
            times.append(time.perf_counter() - t0)
    return q, used_threads, times, results


def parity_word(results, gpu_driver, gpu_exec, gpu_off):
    """Compares the CPU port's placements with the GPU's on the same applications (bit-exact: driver node and, for
    every application that fits, the whole ExecutorNodes slice in order).  -> (applications checked, mismatches)."""
    checked = mism = 0
    for sel, dn, en, off in results:
        gd = np.asarray(gpu_driver)[sel]
        bad = gd != dn
        mism += int(bad.sum())
        checked += len(sel)
        for j in np.nonzero(~bad & (dn >= 0))[0]:
            i = sel[j]
            if not np.array_equal(np.asarray(gpu_exec[gpu_off[i]:gpu_off[i + 1]], dtype=np.int64), en[off[j]:off[j + 1]]):
                mism += 1
    return checked, mism


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, driver, executors, count):
    """Writes the placements of one pack -- what a caller of gp_pack_batch receives -- as float64 .npy files:
    driver_node [apps] and executor_nodes [sum(count)], the latter -1 for applications without a driver node (their
    slots are undefined in the ABI, so they would differ from run to run).  Above DUMP_BYTES in all, executor_nodes is
    a fixed, seeded sample of the slots and executor_nodes_index says which."""
    os.makedirs(out_dir, exist_ok=True)
    driver = np.asarray(driver, dtype=np.float64)
    fits = np.repeat(driver >= 0, count)
    arrays = {"driver_node": driver,
              "executor_nodes": np.where(fits, np.asarray(executors[:len(fits)]), -1).astype(np.float64)}
    room = DUMP_BYTES - driver.nbytes
    if arrays["executor_nodes"].nbytes > room:
        idx = np.sort(np.random.default_rng(0).choice(len(fits), room // 16, replace=False))
        arrays["executor_nodes"] = arrays["executor_nodes"][idx]
        arrays["executor_nodes_index"] = idx.astype(np.float64)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), v)


def common_config(w: dict, q: int, world: int, total_exec: int) -> dict:
    """The `config` object -- identical in the repo arm and the reference arm (same workload, same sizes)."""
    return {"workload": w["desc"], "nodes": w["nodes"], "apps_per_gpu": q, "apps_total": q * world,
            "algo": ALGO_NAME[w["algo"]], "mode": MODE_NAME[w["mode"]], "instance_groups": w["groups"],
            "executors_total_per_gpu": int(total_exec),
            "l2": "256 MiB write between steps, outside the per-step CUDA-event pair (GPU arm); CPU arm: working set > LLC share"}


def calibrated_sample(w: dict, cores: int, budget_s: float, cap: int) -> int:
    """Applications per CPU step so that one step of the literal port takes about `budget_s` seconds on this host
    (the deep-scan workloads run at tens of decisions per second, the headline one at ~10^5)."""
    probe, rate = min(cap, 4 * cores if w["mode"] == 0 else 64), 1.0
    for _ in range(3):
        _, _, times, _ = cpu_reference_run(w, probe, cores, repeats=1)
        rate = probe / max(times[0], 1e-6)
        if times[0] > 0.4 or probe >= cap:
            break
        probe = int(min(cap, max(probe * 8, rate * 0.8)))
    return int(max(min(cap, rate * budget_s), min(cap, 2 * cores)))


def run_reference_arm(args, w):
    """`--impl reference`: the reference's own CPU implementation of the path.  Go cannot run here, so this is the
    literal C restatement of the Go code (oracle/, kind "port") on all host cores, on the repo arm's config.  At N=1 a
    step is the WHOLE workload whenever that takes a few seconds; otherwise (N>1: N x the queue; deep scans) a bounded
    sample, stated in cpu_baseline.sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from k8s_spark_scheduler_b200 import synth
    cores = os.cpu_count() or 1
    _, a, _, _ = make_workload(w, 0)
    q_full = len(a["count"])
    total_exec = int(synth.exec_offsets(a["count"])[-1])
    world = max(args.gpus, 1)
    sample = args.cpu_sample or calibrated_sample(w, cores, 4.0, q_full)     # ~4 s per step -> ~2 min for 25 steps
    q, threads, times, _ = cpu_reference_run(w, sample, cores, repeats=args.steps)
    t = float(np.mean(times))
    value = q / t
    whole = (q == q_full and world == 1)
    line = {
        "impl": "reference", "metric": "gang_placements_per_sec", "value": value, "unit": "decisions/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": common_config(w, q_full, world, total_exec),
        "cpu_baseline": {"value": value, "unit": "decisions/s", "cores": threads, "kind": "port",
                         "sample": (f"the whole workload per step ({q} apps)" if whole else
                                    f"first {q} of the {q_full * world} apps per step") +
                                   ", literal C restatement of the Go path (string-keyed maps, per-candidate map allocation, "
                                   f"ComputePackingEfficiencies on), {threads} host threads; Go toolchain absent so the reference itself cannot run"},
        "e2e": {"value": value, "unit": "decisions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def _watchdog(seconds: float):
    """A hung collective must not hang the caller: hard-exit with an error after `seconds`."""
    def fire():
        print(f"[bench] watchdog: no result after {seconds:.0f} s, aborting", file=sys.stderr, flush=True)
        os._exit(3)
    t = threading.Timer(seconds, fire)
    t.daemon = True
    t.start()
    return t


def load_traffic(kernel_name: str, workload: str):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch from the committed ncu capture (profiles/traffic.json)."""
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        for key, t in json.load(open(tpath)).items():
            if t.get("kernel") == kernel_name and t.get("workload") == workload:
                return t
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="tightly-100k", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-sample", type=int, default=0, help="apps per CPU-baseline step (0 = calibrated to the host)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--wire", default="compact", choices=["compact", "int64"],
                    help="host path layout: compact = what gp_pack_batch_wire allows for this batch; int64 = gp_pack_batch")
    ap.add_argument("--max-seconds", type=float, default=900.0, help="watchdog: abort if the run takes longer")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the placements of the last timed step (rank 0's block) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    wd = _watchdog(args.max_seconds)
    w = WORKLOADS[args.workload]

    if args.impl == "reference":
        run_reference_arm(args, w)
        wd.cancel()
        return

    import torch
    import torch.distributed as dist
    import k8s_spark_scheduler_b200 as g
    if not os.path.exists(g.native.LIB_PATH):      # the benchmark never compiles into the tree it runs from
        raise SystemExit(f"{g.native.LIB_PATH} is missing: build it first (python __graft_entry__.py)")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the library has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    packer = g.GangPacker(device=local_rank, async_snapshot=True)    # one Predicate = snapshot + pack, back to back (GP_CFG_ASYNC_SNAPSHOT)
    stream = torch.cuda.ExternalStream(packer.stream_handle(), device=dev)
    nodes, a, eoff, eorder = make_workload(w, rank)
    q = len(a["count"])
    total_exec = int(a["off"][-1])
    algo, mode = w["algo"], w["mode"]
    n_nodes, n_ord = w["nodes"], len(eorder)

    def dev_t(x, dtype):
        return torch.from_numpy(np.ascontiguousarray(x)).to(dtype).to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ================= value: device-resident inputs, no collective in the data path =====================
    # Every rank holds the snapshot and its own block of the queue in HBM; a step = snapshot layout + pack.
    # (The path shards by application with nothing to exchange while packing; distributing the snapshot and
    #  collecting the placements are the multi-GPU analogue of H2D / D2H and are timed in `e2e` below.)
    # All tensors are allocated on torch's default stream (torch's allocator must never see the library's stream,
    # which dies with the context); only the WORK is enqueued on the library's stream.
    # the snapshot lives in ONE flat buffer so that a single NCCL broadcast can move it (e2e):
    # [cpu int64 x N | mem int64 x N | gpu int64 x N | executor/driver order int32 x len(eorder)]
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
    if mode == 0:
        ta.pop("young")
    d_driver = torch.empty(q, dtype=torch.int32, device=dev)
    d_exec = torch.empty(max(total_exec, 1), dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    torch.cuda.synchronize()

    def device_step():
        packer.set_snapshot_device(tn["cpu"], tn["mem"], tn["gpu"], tn["eoff"], tn["eorder"], tn["eoff"], tn["eorder"])
        packer.pack_batch_device(ta, algo, mode, d_driver, d_exec)

    with torch.cuda.stream(stream):
        # Eager warm-up steps: they also provide the per-kernel times (the library brackets its pack kernel with
        # CUDA events on its own launch stream) and the scan statistics that the roofline object needs.
        pack_ns, prep_ns = [], []
        for _ in range(max(args.warmup, 3)):
            flush.fill_(1)
            device_step()
            st = packer.stats()                # synchronises the stream; reads the pack kernel's own event time
            pack_ns.append(st["pack_kernel_ns"]); prep_ns.append(st["prep_kernel_ns"])
        stats = packer.stats()
        launches_per_step = 4 + int(stats["kernel_launches"])   # build_groups, exec_slots, driver_slots, fill_pair32 + the pack call's own
        # The step is a chain of ~10 small launches; issued from Python its duration depends on how fast the host
        # thread can enqueue them (visibly so with 8 ranks per box).  It is therefore captured ONCE into a CUDA
        # graph and replayed: same kernels, same work, one launch.  BENCH_GRAPH=0 keeps eager launches.
        graph = None
        if os.environ.get("BENCH_GRAPH", "1") != "0":
            try:
                torch.cuda.synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=stream):
                    device_step()
                for _ in range(2):
                    graph.replay()
                torch.cuda.synchronize()
            except Exception as e:   # capture not possible: run eagerly
                print(f"[bench] CUDA graph capture failed ({type(e).__name__}: {e}); running eagerly", file=sys.stderr)
                graph = None
                torch.cuda.synchronize()
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        barrier()
        wall0 = time.perf_counter()
        for s in range(args.steps):
            flush.fill_(s & 0xff)              # L2 flush, outside the event pair
            evs[s][0].record(stream)
            if graph is not None:
                graph.replay()
            else:
                device_step()
            evs[s][1].record(stream)
        barrier()
        wall1 = time.perf_counter()
        step_ms = [e0.elapsed_time(e1) for e0, e1 in evs]
    ms = float(np.mean(step_ms))
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
    value = q * world / (ms * 1e-3)
    dev_driver_np = d_driver.cpu().numpy()          # device-resident results: the N>1 parity word compares the host path with them
    dev_exec_np = d_exec.cpu().numpy()

    # ================= e2e: host buffers in, host results out ================================================
    # all-zero GPU request columns are passed as NULL (= 0), as the ABI allows; the shim knows while marshalling
    # Wire format, chosen per batch like the shim would (include/gangpack.h, gp_pack_batch_wire): int32 millicores / MiB
    # when every quantity is exactly representable, offsets derived on the device and uint16 node indices for the
    # independent tightly-pack / distribute-evenly path on <= 65 535 nodes; --wire int64 keeps the plain gp_pack_batch layout.
    fused = (mode == 0 and algo != 2)
    wire = None
    src = a
    if args.wire == "compact":
        c32 = g.native.compact_apps({k: a[k] for k in ("drv_cpu", "drv_mem", "drv_gpu", "exe_cpu", "exe_mem", "exe_gpu")}, mem_shift=20)
        wire = dict(quantity_bits=32 if c32 is not None else 64, mem_shift=20,
                    node_bits=16 if (fused and n_nodes <= 65535) else 32, offsets=not fused)
        if c32 is not None:
            src = dict(a); src.update(c32)
    host_keys = [k for k in src if not (k in ("drv_gpu", "exe_gpu") and not a[k].any())]
    if wire is not None and not wire["offsets"]:
        host_keys.remove("off")
    q_cols = [k for k in ("drv_cpu", "drv_mem", "exe_cpu", "exe_mem", "drv_gpu", "exe_gpu") if k in host_keys]
    pin = packer.pinned_columns(q, q_cols, dtype=src["drv_cpu"].dtype)   # one pinned block, column after column (as the shim allocates it)
    for k in host_keys:
        if k not in pin:
            pin[k] = packer.pinned(len(src[k]), src[k].dtype)
        pin[k][:] = src[k]
    if w["groups"] == 1:
        pin.pop("group", None)
    if mode == 0:
        pin.pop("young", None)
    # the snapshot SoA also lives in pinned host memory (what the shim fills per Predicate)
    pn = {}
    for k, v in (("cpu", nodes["avail_cpu"]), ("mem", nodes["avail_mem"]), ("gpu", nodes["avail_gpu"]),
                 ("eorder", eorder), ("eoff", eoff)):
        pn[k] = packer.pinned(len(v), v.dtype); pn[k][:] = v
    snap_bytes = 3 * 8 * n_nodes + 2 * 4 * n_ord + 2 * 4 * len(eoff)
    in_bytes = sum(v.nbytes for v in pin.values())
    shm = None

    if world == 1:
        node_dt = np.uint16 if (wire and wire["node_bits"] == 16) else np.int32
        out_driver = packer.pinned(q, np.int32)
        out_exec = packer.pinned(max(total_exec, 1), node_dt)
        h2d = in_bytes + snap_bytes
        d2h = out_driver.nbytes + out_exec.itemsize * total_exec

        # the argument structs are marshalled once over the long-lived pinned buffers, like a shim does; a step = two FFI calls
        wire_eff = wire or dict(quantity_bits=64, node_bits=32, offsets=True)
        call_snapshot = packer.bind_snapshot(pn["cpu"], pn["mem"], pn["gpu"], pn["eorder"], pn["eorder"], pn["eoff"], pn["eoff"])
        call_pack = packer.bind_batch(pin, algo, mode, (out_driver, out_exec), wire_eff)

        def e2e_step():
            call_snapshot()
            call_pack()
            return int(out_driver[0])          # the host reads the result

        e2e_step_desc = "gp_set_snapshot + gp_pack_batch_wire from pinned host buffers to host results"
        snap_launches = 4
    else:
        # N>1 (SURVEY 8e).  ONE scheduler process (rank 0) owns the cluster state and consumes every placement; one worker
        # process per GPU.  Rank 0 uploads the snapshot (H2D) and ONE NCCL broadcast distributes it over NVLink; every rank
        # packs its own host-resident block of the queue and copies ITS placements over ITS OWN PCIe link straight into the
        # scheduler's result buffer -- a POSIX shared-memory segment page-locked by every worker (gp_register_host).  No
        # gather through one GPU, no collective on the results.  Wall clock between barriers, max over ranks.
        from k8s_spark_scheduler_b200 import multigpu
        node_dt = np.uint16 if (wire and wire["node_bits"] == 16) else np.int32
        shm = multigpu.SharedResults(f"gangpack_bench_{os.environ.get('MASTER_PORT', '0')}", q, total_exec, node_dt, device=dev)
        packer.register_host(shm.mine)
        out_driver, out_exec = shm.driver, shm.executors
        h_snap = torch.empty(snapbuf.numel(), dtype=torch.int64).pin_memory()
        h_snap.copy_(snapbuf.cpu())
        h2d = in_bytes + (snapbuf.numel() * 8 if rank == 0 else 0)
        d2h = out_driver.nbytes + out_exec.itemsize * total_exec

        call_pack = packer.bind_batch(pin, algo, mode, (out_driver, out_exec), wire or dict(quantity_bits=64, node_bits=32, offsets=True))

        def e2e_step():
            with torch.cuda.stream(stream):
                if rank == 0:
                    snapbuf.copy_(h_snap, non_blocking=True)
                multigpu.broadcast_snapshot(snapbuf, src=0)
                packer.set_snapshot_device(tn["cpu"], tn["mem"], tn["gpu"], tn["eoff"], tn["eorder"], tn["eoff"], tn["eorder"])
            call_pack()
            return int(out_driver[0])

        e2e_step_desc = ("rank 0 H2D snapshot + ONE NCCL broadcast (NVLink) + layout; every rank: gp_pack_batch from its pinned host "
                         "block of the queue, results DMA'd over its own PCIe link into the scheduler's shared-memory result buffer")
        snap_launches = 4

    for _ in range(max(args.warmup, 3)):
        e2e_step()
    barrier()
    e2e_t = []
    e2e_launches = 0
    for s in range(args.steps):
        with torch.cuda.stream(stream):
            flush.fill_(s & 0xff)
        stream.synchronize()
        if world > 1:
            barrier()                      # ranks start the step together (outside the timed region)
        t0 = time.perf_counter()
        e2e_step()                         # returns when this rank's placements are in host memory
        e2e_t.append(time.perf_counter() - t0)
        e2e_launches += snap_launches + packer.stats()["kernel_launches"]   # snapshot layout + the pack call's launches (per pipelined chunk)
    e2e_ms = float(np.mean(e2e_t)) * 1e3
    if world > 1:
        t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_value = q * world / (e2e_ms * 1e-3)
    clocks = sampler.stop() if rank == 0 else None

    # ---- parity word (outside every timed region) ------------------------------------------------------
    # (a) every rank: the host path's placements == the device-resident path's placements, all q applications
    # (FIFO modes included: both ran the same queue against the same snapshot);
    fits = dev_driver_np >= 0
    emask = np.repeat(fits, a["count"])
    path_mism = int((np.asarray(out_driver) != dev_driver_np).sum()) + \
        int((np.asarray(out_exec[:total_exec])[emask] != dev_exec_np[:total_exec][emask]).sum())
    if world > 1:
        t = torch.tensor([path_mism], device=dev, dtype=torch.int64); dist.all_reduce(t); path_mism = int(t.item())
        # (b) rank 0 -- the consumer -- finds every rank's block in the shared buffer: each rank publishes a checksum of the
        # placements it computed on the device, rank 0 recomputes them from the shared segment
        dist.barrier()
        mine_sum = torch.tensor([int(dev_driver_np.astype(np.int64).sum()), int(dev_exec_np[:total_exec][emask].astype(np.int64).sum())],
                                device=dev, dtype=torch.int64)
        sums = [torch.zeros(2, device=dev, dtype=torch.int64) for _ in range(world)]
        dist.all_gather(sums, mine_sum)
        if rank == 0:
            for r in range(1, world):
                rd, _ = shm.block(r)
                if int(rd.astype(np.int64).sum()) != int(sums[r][0].item()):
                    path_mism += 1
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dev_driver_np, dev_exec_np, a["count"])

    # ---- roofline of the dominant kernel (pack) ----------------------------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"]); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak = 6650.0; peak_src = "fallback (B200_PROFILING.md 6.65 TB/s)"
    R = 2   # cpu + mem; the gpu array is skipped when no request and no negative availability (DESIGN.md)
    k_total = total_exec
    # scan path: 8R bytes per node evaluated; table path: one 4-byte prefix word per probe; per driver candidate its slot
    # index + its (cpu, mem) record; per application the tuple (64 B) + the result header (8 B); 4 B per emitted executor
    scan_nodes = stats["scan_path_nodes"] if fused else stats["nodes_scanned"]
    table_probes = stats["nodes_scanned"] - scan_nodes
    alg_bytes = (scan_nodes * 8 * R + table_probes * 4 + stats["drivers_tried"] * (4 + 16 if fused else 4)
                 + q * (64 + 8) + 4 * k_total)
    nominal_bytes = q * (w["nodes"] * 8 * R + w["nodes"] * 4 + 64 + 8) + 4 * k_total
    pack_s = float(np.mean(pack_ns)) * 1e-9
    tables_on = fused and os.environ.get("GANGPACK_TABLES", "1") != "0"
    kernel_name = (("gp_decide_tables" if tables_on else "gp_pack_listed") if fused else
                   ("gp_pack_independent" if mode == 0 else "gp_pack_fifo_cta")) + f"<{ALGO_NAME[algo]}>"
    tr = load_traffic(kernel_name, args.workload) if world == 1 else None
    traffic = tr["dram_bytes_per_launch"] if tr else None
    roofline = {
        # `achieved`/`frac` follow SURVEY 8(d): ALGORITHMIC bytes / kernel time against the measured HBM copy bandwidth.
        # The kernel itself is NOT limited by DRAM: `limiter` says what ncu shows, `dram_frac` what the DRAM pins really carry.
        "bound": "hbm", "kernel": kernel_name,
        "achieved": alg_bytes / pack_s / 1e9, "peak": peak, "unit": "GB/s",
        "frac": alg_bytes / pack_s / 1e9 / peak, "peak_source": peak_src,
        "traffic": traffic,
        "dram_frac": (traffic / pack_s / 1e9 / peak) if traffic else None,
        "limiter": (tr or {}).get("limiter", "instruction issue / L1 latency (integer scan over an L1/L2-resident snapshot); see DESIGN.md section 6"),
        "algorithmic_bytes_per_launch": int(alg_bytes), "kernel_ms": pack_s * 1e3,
        "nodes_scanned_per_decision": scan_nodes / q, "table_words_per_decision": table_probes / q,
        "drivers_tried_per_decision": stats["drivers_tried"] / q, "scan_path_apps": int(stats["scan_path_apps"]),
        "full_table_equivalent_GBps": nominal_bytes / pack_s / 1e9,
        "note": "algorithmic bytes use the nodes actually visited (early exit is exact); the snapshot is served "
                "from L1/L2, so DRAM traffic is far below this -- dram_frac is the honest HBM share",
    }

    # ---- CPU baseline on the box's host cores (rank 0, N=1 only) + parity of the GPU results against it -----
    cpu_baseline = None
    parity_checked = parity_mism = 0
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        sample = args.cpu_sample or calibrated_sample(w, cores, 12.0, q)          # ~10-20 s of CPU work
        qs, threads, times, results = cpu_reference_run(w, sample, cores, repeats=1)
        cpu_baseline = {"value": qs / times[0], "unit": "decisions/s", "cores": threads, "kind": "port",
                        "sample": f"first {qs} apps of the workload, literal C restatement of the Go path (string-keyed maps, "
                                  f"per-candidate map allocation, ComputePackingEfficiencies on), {threads} threads, "
                                  f"{times[0]:.2f} s"}
        parity_checked, parity_mism = parity_word(results, out_driver, out_exec, a["off"])

    if rank == 0:
        cfg = common_config(w, q, world, total_exec)
        cfg.update({"step": "snapshot layout + pack, device-resident inputs, no collective in the data path "
                            "(every rank packs its own block of the queue against its copy of the snapshot); "
                            + ("the launch chain is replayed from one CUDA graph" if graph is not None else "eager launches"),
                    "e2e_step": e2e_step_desc, "e2e_wire": wire or "int64 quantities, int64 offsets, int32 node indices",
                    "decision_path": ("per-shape capacity tables" if (fused and os.environ.get("GANGPACK_TABLES", "1") != "0") else "node-order scan")
                                     + f"; {stats['scan_path_apps']} of {q} applications decided by the scan"})
        line = {
            "metric": "gang_placements_per_sec", "value": value, "unit": "decisions/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": cfg,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "decisions/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": launches_per_step * args.steps + e2e_launches,
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "parity_checked": int(parity_checked), "mismatches": int(parity_mism),
            "parity": {"vs_cpu_port": {"apps": int(parity_checked), "mismatches": int(parity_mism)},
                       "host_path_vs_device_path": {"apps": q * world, "mismatching_words": path_mism}},
            "kernel_ms": {"pack": pack_s * 1e3, "prep": float(np.mean(prep_ns)) * 1e-6},
            "wall_s_value_region": wall1 - wall0,
        }
        print(json.dumps(line), flush=True)

    # ---- orderly teardown: the driver's exit hook must see this process with libgangpack.so mapped -------
    # Everything torch used on the library's stream (device tensors, the pinned snapshot copy -- torch's host allocator
    # records an event on that stream when the block is freed) and every view into the shared segment goes BEFORE gp_destroy.
    torch.cuda.synchronize()
    del graph, evs
    del snapbuf, tn, ta, d_driver, d_exec, flush
    h_snap = e2e_step = rd = sums = mine_sum = t = None
    pin = pn = out_driver = out_exec = None
    call_pack = call_snapshot = None
    import gc
    gc.collect()
    torch.cuda.synchronize()
    packer.close()                                    # frees pinned blocks, unregisters the shared segment, gp_destroy
    if shm is not None:
        shm.close()
    if world > 1:
        dist.destroy_process_group()
    wd.cancel()
    if (parity_mism or path_mism) and rank == 0:
        raise SystemExit(f"parity failure: {parity_mism} vs the CPU port, {path_mism} host-path vs device-path")


if __name__ == "__main__":
    main()
