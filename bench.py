#!/usr/bin/env python
"""bench.py — scans/s of the per-scan road/curb classification path (BASELINE.json metric) on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W]                 our CUDA path (liburf_b200.so through the C-ABI)
  python bench.py --impl reference [--gpus N] [--steps K] [--warmup W] the reference's own CPU implementation, host cores
  python bench.py ... --dump-outputs DIR                               also writes what the last timed step computed
                                                                       (dump_outputs), to compare two builds

A "step" is one pass of the hot path over one batch of `--batch` distinct synthetic OS1-64 scans (BASELINE config 2:
64 rings x 2048 columns = 131,072 points per scan, all three detectors + blindSpots, full-ROI preset so every point
takes part). N > 1 is launched by torchrun (one rank per GPU); scans are independent units, so ranks just process their
own batches (weak scaling, no data-path collective) and NCCL carries only the barrier and the max-over-ranks time.

One JSON line on stdout (rank 0): value = whole-job scans/s with inputs resident in HBM, timed with CUDA events on the
library's stream; e2e = the same metric through urf_process_batch with pinned HOST buffers (H2D + D2H inside the timed
region); roofline = the dominant kernel's algorithmic bytes / its CUDA-event duration vs the measured HBM peak;
cpu_baseline = the reference's CPU path timed on this box's host cores on a bounded sample.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from urban_road_filter_b200 import FULL_ROI, UrfResult, make_params  # noqa: E402
from urban_road_filter_b200.shard import allreduce_max, allreduce_sum, seeds_for_rank  # noqa: E402
from urban_road_filter_b200.synth import SHAPES, make_scan  # noqa: E402

ALGO_BYTES_PER_POINT = 20          # SURVEY.md §8(d): 16 B float4 read + 4 B int32 label written, per input point
FALLBACK_HBM_GBS = 6650.0          # /opt/skills/guides/B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent


_ABLATION = {}          # detector switches of BASELINE config 5 (--no-star / --no-xzero / --no-zzero), shared with the CPU workers


def bench_params(shape_key: str):
    sh = SHAPES[shape_key]
    return make_params(channels=sh.channels, interval=sh.interval, **_ABLATION, **FULL_ROI)


def workload_config(shape_key: str) -> dict:
    """The `config` block, identical for both arms: it names the workload, nothing that depends on who runs it."""
    sh = SHAPES[shape_key]
    n = sh.rings * sh.cols
    return {"workload": f"{sh.name} {n}-pt scans, {detectors_text()}, full-ROI preset (BASELINE config {shape_key[1:]})",
            "shape": shape_key, "points_per_scan": n, "rings": sh.rings, "channels": sh.channels, "interval": sh.interval}


def detectors_text() -> str:
    on = [name for name, key in (("star", "star_shaped_method"), ("x_zero", "x_zero_method"), ("z_zero", "z_zero_method"))
          if _ABLATION.get(key, 1)]
    return ("all three detectors" if len(on) == 3 else ("detectors: " + "+".join(on) if on else "no curb detector")) + " + blindSpots"


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation (oracle/_ref = unmodified reference sources; else the oracle port).
# One single-threaded process per host core (the reference is single-threaded by construction, src/main.cpp:54), each
# with its own scan; the pool and the scans persist across steps so that a step only contains filtered() calls.
_W = {}


def _cpu_init(shape_key, seed0, use_ref, counter, ablation=None):
    sys.path.insert(0, ROOT)
    _ABLATION.update(ablation or {})
    from oracle.pyoracle import PortOracle, RefOracle
    with counter.get_lock():
        wid = counter.value
        counter.value += 1
    _W["pts"] = make_scan(shape_key, seed0 + wid)
    _W["prm"] = bench_params(shape_key)
    _W["orc"] = RefOracle() if use_ref else PortOracle()
    _W["orc"].time(_W["pts"], _W["prm"], 1)          # untimed first call: page-faults the reference's big allocations


def _cpu_step(repeat):
    return _W["orc"].time(_W["pts"], _W["prm"], repeat), repeat


class CpuReference:
    def __init__(self, shape_key: str, workers: int, seed0: int = 10_000):
        import multiprocessing as mp
        from oracle.pyoracle import RefOracle
        self.use_ref = RefOracle.available()
        self.workers = workers
        ctx = mp.get_context("fork" if not _cuda_initialised() else "spawn")
        self.pool = ctx.Pool(workers, initializer=_cpu_init, initargs=(shape_key, seed0, self.use_ref, ctx.Value("i", 0), dict(_ABLATION)))
        self.pool.map(_cpu_step, [0] * workers)          # make sure every worker is initialised

    @property
    def kind(self) -> str:
        return "reference" if self.use_ref else "port"

    def step(self, repeat: int = 1):
        """Aggregate scans/s of all workers running `repeat` scans each at the same time, and the median ms per scan."""
        res = self.pool.map(_cpu_step, [repeat] * self.workers, chunksize=1)
        return sum(r / s for s, r in res), 1e3 * statistics.median(s / r for s, r in res)

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_reference_rate(shape_key: str, workers: int, repeat: int, seed0: int = 10_000):
    ref = CpuReference(shape_key, workers, seed0)
    try:
        rate, per_scan_ms = ref.step(repeat)
    finally:
        ref.close()
    return rate, per_scan_ms, ref.kind


def _cuda_initialised() -> bool:
    try:
        import torch
        return torch.cuda.is_initialized()
    except Exception:
        return False


def usable_cores(shape_key: str = "C2") -> int:
    """One single-threaded reference process per host core, capped by memory: the reference allocates
    channels x N x 48 B per scan (lidar_segmentation.cpp:207) — 0.4 GB at C2, 12.9 GB at C5."""
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    sh = SHAPES[shape_key]
    per_proc = 1.5 * sh.channels * sh.rings * sh.cols * 48 + 2**30
    try:
        import psutil
        cores = min(cores, max(1, int(psutil.virtual_memory().available / per_proc)))
    except Exception:
        pass
    return max(1, cores)


# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled in the background (recipe of B200_PROFILING.md)."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for _, r in self.rows]
        sm, mx, reasons = [], [], set()
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[2])); mx.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v == "Active":
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def pin_to_gpu_numa_node(torch, local: int) -> None:
    """Run this rank on the CPUs of the NUMA node its GPU hangs off (sysfs), so that pinned host buffers and the copy
    threads are local to the PCIe root of the GPU. Best effort: silently does nothing where sysfs says nothing."""
    try:
        pr = torch.cuda.get_device_properties(local)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return
        cpus: set[int] = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:
        pass


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel: str):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture, if one is recorded."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(kernel)
        except Exception:
            return None
    return None


DUMP_MAX_LABELS = 1 << 23          # 32 MiB of float32 labels per process; larger outputs are sampled
COUNT_FIELDS = ("status", "n_in", "n_roi", "n_rings", "n_order", "n_road", "n_curb", "n_vert", "flags")


def dump_outputs(path: str, labels, outs, rank: int, world: int) -> None:
    """Writes what one device-resident step returned to its caller, so two builds can be compared output for output:
    label.npy  float32 labels of the (batch, points) label array, flattened; all of them when there are at most
               DUMP_MAX_LABELS / world, else that many at flat positions drawn with seed 0 (the same for the same arguments);
    counts.npy float64 (batch, 9): the per-scan counts of urf_result (COUNT_FIELDS);
    vert.npy   float32 (batch, URF_MAX_VERTS, 4): the marker candidate vertices, rows past n_vert zeroed.
    With several ranks each writes its own files, suffixed _rank<r>."""
    import torch
    os.makedirs(path, exist_ok=True)
    sfx = f"_rank{rank}" if world > 1 else ""
    flat = labels.reshape(-1)
    cap = DUMP_MAX_LABELS // world
    if flat.numel() > cap:
        idx = np.sort(np.random.default_rng(0).choice(flat.numel(), size=cap, replace=False))
        flat = flat[torch.from_numpy(idx).to(flat.device)]
    np.save(os.path.join(path, f"label{sfx}.npy"), flat.cpu().numpy().astype(np.float32))
    np.save(os.path.join(path, f"counts{sfx}.npy"), np.array([[getattr(o, f) for f in COUNT_FIELDS] for o in outs], np.float64))
    vert = np.stack([np.ctypeslib.as_array(o.vert).copy() for o in outs]).astype(np.float32)
    for b, o in enumerate(outs):
        vert[b, o.n_vert:] = 0.0
    np.save(os.path.join(path, f"vert{sfx}.npy"), vert)


# ----------------------------------------------------------------------------------------------------------------------
def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0            # the reference arm is a host-CPU measurement: rank 0 alone runs and prints it
    cores = usable_cores(args.shape)
    n = SHAPES[args.shape].rings * SHAPES[args.shape].cols
    single_rate, single_ms, _ = cpu_reference_rate(args.shape, 1, 2, seed0=30_000)
    ref = CpuReference(args.shape, cores, seed0=20_000)
    kind = ref.kind
    for _ in range(args.warmup):
        ref.step(1)
    t0 = time.perf_counter()
    rates = [ref.step(1)[0] for _ in range(args.steps)]
    wall = time.perf_counter() - t0
    ref.close()
    value = statistics.median(rates)
    line = {
        "impl": "reference", "metric": "scans_per_sec", "value": value, "unit": "scans/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32/f64", "data": "synthetic",
        "config": workload_config(args.shape),
        "step": f"{cores} scans, one per host core (one single-threaded process each: the reference is single-threaded, src/main.cpp:54)",
        "mpoints_per_sec": value * n / 1e6,
        "cpu_baseline": {"value": value, "unit": "scans/s", "cores": cores, "kind": kind,
                         "sample": f"{cores} single-threaded processes x 1 scan per step, median of {args.steps} steps",
                         "single_process": {"value": single_rate, "unit": "scans/s", "ms_per_scan": single_ms, "cores": 1,
                                            "sample": "1 process x 2 scans after one untimed scan"}},
        "e2e": {"value": value, "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="default: 200 (urf), 10 (reference)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="urf", choices=["urf", "reference"])
    ap.add_argument("--batch", type=int, default=128, help="scans per step and per GPU")
    ap.add_argument("--shape", default="C2", choices=sorted(SHAPES))
    ap.add_argument("--cpu-repeat", type=int, default=3, help="scans per host core in the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--groups", type=int, default=0, help="compute streams per device-resident batch (0 = library default)")
    ap.add_argument("--no-e2e", action="store_true", help="tuning runs: skip the host-buffer region")
    ap.add_argument("--sub", type=int, default=-1, help="scans per sub-batch of a device-resident step (library option 5)")
    ap.add_argument("--graph", type=int, default=-1, help="replay a device-resident step as one CUDA graph (library option 6)")
    ap.add_argument("--reuse", type=int, default=-1, help="sub-batches of a stream share a workspace slot (library option 7)")
    ap.add_argument("--rd", type=int, default=-1, help="k_ring_detect variant (library option 8: 8, 6, 5 or 4 = four positions per thread)")
    ap.add_argument("--mk", type=int, default=-1, help="marker search variant (library option 9: 0 cluster of 8 CTAs, 1 one CTA per scan)")
    ap.add_argument("--sweep", default="", help="tuning: ';'-separated groups,sub,graph,reuse settings timed one after the other")
    ap.add_argument("--no-star", action="store_true", help="detector ablation (BASELINE config 5): star_shaped_method off")
    ap.add_argument("--no-xzero", action="store_true", help="detector ablation: x_zero_method off")
    ap.add_argument("--no-zzero", action="store_true", help="detector ablation: z_zero_method off")
    ap.add_argument("--no-with-order", action="store_true", help="skip the second timed pass that also produces the emission order")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the labels (sampled above 2^23), per-scan counts and vertices of the "
                         "last device-resident step as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "urf" else args.warmup
    if args.steps is None:
        args.steps = 200 if args.impl == "urf" else 10
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "urf" or args.sweep):
        ap.error("--dump-outputs writes the outputs of the timed device-resident path: not with --impl reference or --sweep")
    for flag, key in ((args.no_star, "star_shaped_method"), (args.no_xzero, "x_zero_method"), (args.no_zzero, "z_zero_method")):
        if flag:
            _ABLATION[key] = 0

    if args.impl == "reference":
        return run_reference_arm(args)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    # CPU baseline first (rank 0, N == 1 only), before CUDA is initialised in this process
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = usable_cores(args.shape)
        # (i) ONE process alone on the box: the stable anchor (the reference node is single-threaded, src/main.cpp:54);
        # (ii) one process per core, which on some hosts is bound by page faults on the reference's channels x N x 48 B array
        single_rate, single_ms, _ = cpu_reference_rate(args.shape, 1, 2)
        rate, per_scan_ms, kind = cpu_reference_rate(args.shape, cores, args.cpu_repeat)
        cpu_baseline = {"value": rate, "unit": "scans/s", "cores": cores, "kind": kind,
                        "single_process": {"value": single_rate, "unit": "scans/s", "ms_per_scan": single_ms, "cores": 1,
                                           "sample": "1 process x 2 scans after one untimed scan"},
                        "sample": f"{cores} single-threaded processes x {args.cpu_repeat} scans each (after one untimed scan), "
                                  f"median {per_scan_ms:.0f} ms per scan per core"}

    import torch
    import torch.distributed as dist
    from urban_road_filter_b200 import api

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl urf needs a CUDA device: urban_road_filter_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    pin_to_gpu_numa_node(torch, local)      # before any pinned allocation: host buffers land next to this rank's GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    sh = SHAPES[args.shape]
    B, n = args.batch, sh.rings * sh.cols
    prm = bench_params(args.shape)
    clouds = [make_scan(args.shape, seed) for seed in seeds_for_rank(B, rank)]
    det = api.Detector(max_points=n, max_batch=B, device=local, params=prm)
    if args.groups:
        det.set_option(2, args.groups)
    for opt, v in ((5, args.sub), (6, args.graph), (7, args.reuse), (8, args.rd), (9, args.mk)):
        if v >= 0:
            det.set_option(opt, v)
    lib, ctx = det.lib, det._ctx
    S = n
    x = torch.empty((B, S, 4), dtype=torch.float32, device="cuda")
    for b, c in enumerate(clouds):
        x[b].copy_(torch.from_numpy(c))
    labels = torch.empty((B, S), dtype=torch.int32, device="cuda")
    ns = (C.c_int * B)(*([n] * B))
    outs = (UrfResult * B)()
    stream = torch.cuda.ExternalStream(lib.urf_stream(ctx), device=torch.device("cuda", local))

    def step_device():
        rc = lib.urf_enqueue_batch_device(ctx, x.data_ptr(), S, ns, B, labels.data_ptr())
        assert rc == 0, lib.urf_last_cuda_error(ctx)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(args.warmup):
        step_device()
    assert lib.urf_finish_batch_device(ctx, outs) == 0
    if args.sweep:                       # tuning: scheduling settings of the device-resident step, same process, same data
        ref_road = sum(o.n_road for o in outs)
        for cfg in args.sweep.split(";"):
            f = [int(v) for v in cfg.split(",")]
            g, sub, graph, reuse = f[:4]
            det.set_option(2, g); det.set_option(5, sub); det.set_option(6, graph); det.set_option(7, reuse)
            if len(f) > 4:
                det.set_option(8, f[4])                 # k_ring_detect variant
            if len(f) > 5:
                det.set_option(9, f[5])                 # marker search: cluster (0) or one CTA per scan (1)
            if len(f) > 6:
                det.set_option(10, f[6])                # near-first pivot rank among 32 samples
            if len(f) > 7:
                det.set_option(11, f[7])                # ring detector on a side stream next to the star-shaped search
            if len(f) > 8:
                det.set_option(12, f[8])                # widest single-warp star sort network: 32 or 16 elements per lane
            for _ in range(3):
                step_device()
            torch.cuda.synchronize()
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            a.record(stream)
            for _ in range(args.steps):
                step_device()
            b_.record(stream)
            t_enq = time.perf_counter() - t0
            torch.cuda.synchronize()
            assert lib.urf_finish_batch_device(ctx, outs) == 0
            ok = sum(o.n_road for o in outs) == ref_road
            print(json.dumps({"sweep": cfg, "ms_per_step": a.elapsed_time(b_) / args.steps, "enqueue_ms_per_step": 1e3 * t_enq / args.steps,
                              "launches": det.last_launch_count(), "road_ok": ok}), flush=True)
        det.close()
        return 0
    # ---- timed region 1: inputs resident in HBM; K steps enqueued back to back, no host sync inside. The library spreads
    # ---- the batch over 2 compute streams (independent scans), joined on its main stream, where the events are recorded.
    ktimes: dict[str, float] = {}
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_w0 = time.time()
    e0.record(stream)
    for _ in range(args.steps):
        step_device()
    e1.record(stream)
    barrier()
    t_w1 = time.time()
    dev_ms = e0.elapsed_time(e1)
    assert lib.urf_finish_batch_device(ctx, outs) == 0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, labels, outs, rank, world)
    launches = det.last_launch_count() * args.steps
    n_road = sum(o.n_road for o in outs)
    # ---- timed region 1w: the same K steps with the per-ring azimuth sort (lidar_segmentation.cpp:289-291) and the emission
    # ---- order written to HBM: what the node needs to publish its clouds, on top of labels + vertices
    with_order = None
    if not args.no_with_order:
        order = torch.empty((B, S), dtype=torch.int32, device="cuda")

        def step_order():
            rc = lib.urf_enqueue_batch_device_ex(ctx, x.data_ptr(), S, ns, B, labels.data_ptr(), order.data_ptr())
            assert rc == 0, lib.urf_last_cuda_error(ctx)

        for _ in range(3):
            step_order()
        barrier()
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record(stream)
        for _ in range(args.steps):
            step_order()
        w1.record(stream)
        barrier()
        with_order = {"dev_ms": w0.elapsed_time(w1)}
        assert lib.urf_finish_batch_device(ctx, outs) == 0
        assert sum(o.n_road for o in outs) == n_road
        det.set_option(1, 3)                 # three more steps on one stream with per-kernel events: what the order costs
        for _ in range(3):
            step_order()
        assert lib.urf_finish_batch_device(ctx, outs) == 0
        okt: dict[str, float] = {}
        for slot in range(3):
            for name, ms in det.kernel_times(slot):
                okt[name] = okt.get(name, 0.0) + ms / 3
        det.set_option(1, 0)
        with_order["kernel_ms"] = {k: okt[k] for k in ("k_sort_rings", "k_scatter") if k in okt}
        del order
    # ---- timed region 1b: the same steps once more on ONE stream with a CUDA event in front of every kernel (per-kernel
    # ---- durations are only meaningful without inter-stream overlap); feeds the roofline block, not `value`
    kprof = min(args.steps, 5)
    det.set_option(1, kprof)
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record(stream)
    for _ in range(kprof):
        step_device()
    pe1.record(stream)
    assert lib.urf_finish_batch_device(ctx, outs) == 0
    serial_ms = pe0.elapsed_time(pe1) / kprof
    for slot in range(kprof):
        for name, ms in det.kernel_times(slot):
            ktimes[name] = ktimes.get(name, 0.0) + ms / kprof
    det.set_option(1, 0)
    # ---- timed region 2: end to end through the host-buffer C-ABI call ---------------------------------------------
    if args.no_e2e:
        if rank == 0:
            print(json.dumps({"tuning": True, "groups": args.groups, "ms_per_step": dev_ms / args.steps, "serial_ms_per_step": serial_ms,
                              "kernel_ms": {k: round(v, 4) for k, v in sorted(ktimes.items(), key=lambda kv: -kv[1])}}), flush=True)
        det.close()
        if world > 1:
            dist.destroy_process_group()
        return 0
    h_in = [torch.from_numpy(c).pin_memory() for c in clouds]
    h_lab = [torch.empty(n, dtype=torch.int32).pin_memory() for _ in range(B)]
    ptrs = (C.c_void_p * B)(*[t.data_ptr() for t in h_in])
    res = (UrfResult * B)()
    for b in range(B):
        res[b].label = C.cast(h_lab[b].data_ptr(), C.POINTER(C.c_int32))

    def step_e2e():
        rc = lib.urf_process_batch(ctx, ptrs, ns, B, res)
        assert rc == 0, lib.urf_last_cuda_error(ctx)

    for _ in range(args.warmup):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    # ---- what PCIe alone costs for these buffers: the same pinned arrays copied H2D / D2H with nothing else going on
    d_tmp = torch.empty((B, S, 4), dtype=torch.float32, device="cuda")
    d_lab = torch.empty((B, S), dtype=torch.int32, device="cuda")
    h_scratch = [torch.empty(n, dtype=torch.int32).pin_memory() for _ in range(4)]      # not h_lab: its contents are compared below
    pe = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    cs = torch.cuda.Stream()
    with torch.cuda.stream(cs):
        for rep in range(2):
            pe[0].record(cs)
            for b in range(B):
                d_tmp[b, :n].copy_(h_in[b], non_blocking=True)
            pe[1].record(cs)
            pe[2].record(cs)
            for b in range(B):
                h_scratch[b % 4].copy_(d_lab[b, :n], non_blocking=True)
            pe[3].record(cs)
        cs.synchronize()
    h2d_ms, d2h_ms = pe[0].elapsed_time(pe[1]), pe[2].elapsed_time(pe[3])
    # both directions at once (what an e2e step asks of the link): H2D on one stream, D2H on another, until both are done
    cs2 = torch.cuda.Stream()
    be = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    torch.cuda.synchronize()
    be[0].record(cs)
    cs2.wait_event(be[0])
    with torch.cuda.stream(cs):
        for b in range(B):
            d_tmp[b, :n].copy_(h_in[b], non_blocking=True)
        be[1].record(cs)
    with torch.cuda.stream(cs2):
        for b in range(B):
            h_scratch[b % 4].copy_(d_lab[b, :n], non_blocking=True)
        be[2].record(cs2)
    torch.cuda.synchronize()
    bidir_ms = max(be[0].elapsed_time(be[1]), be[0].elapsed_time(be[2]))
    del d_tmp, d_lab
    # ---- the lean entry point (opt-in ABI addition): packed xyz in (12 B/pt), int8 labels out (1 B/pt), same results
    h_xyz = [torch.from_numpy(np.ascontiguousarray(c[:, :3])).pin_memory() for c in clouds]
    h_l8 = [torch.empty(n, dtype=torch.int8).pin_memory() for _ in range(B)]
    xptrs = (C.c_void_p * B)(*[t.data_ptr() for t in h_xyz])
    l8ptrs = (C.c_void_p * B)(*[t.data_ptr() for t in h_l8])
    res_lean = (UrfResult * B)()

    def step_lean():
        rc = lib.urf_process_batch_xyz(ctx, xptrs, ns, B, res_lean, l8ptrs)
        assert rc == 0, lib.urf_last_cuda_error(ctx)

    for _ in range(args.warmup):
        step_lean()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_lean()
    torch.cuda.synchronize()
    lean_ms = (time.perf_counter() - t0) * 1e3
    barrier()
    assert sum(r.n_road for r in res_lean) == n_road, "lean and default host paths disagree"
    assert all(bool((h_l8[b].to(torch.int32) == h_lab[b]).all()) for b in range(0, B, max(1, B // 4))), "int8 labels differ from the int32 ones"
    if with_order is not None:               # the same call with res[b].order set: the order comes back too (+4 B per point)
        h_ord = [torch.empty(n, dtype=torch.int32).pin_memory() for _ in range(B)]
        for b in range(B):
            res[b].order = C.cast(h_ord[b].data_ptr(), C.POINTER(C.c_int32))
        for _ in range(2):
            step_e2e()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_e2e()
        torch.cuda.synchronize()
        with_order["e2e_ms"] = (time.perf_counter() - t0) * 1e3
        barrier()
        for b in range(B):
            res[b].order = None
    t_w2 = time.time()
    clocks = sampler.stop(t_w0, t_w2) if sampler else None
    print(f"[rank {rank}] device {dev_ms / args.steps:.3f} ms/step, e2e {1e3 * e2e_s / args.steps:.3f} ms/step", file=sys.stderr)
    assert sum(r.n_road for r in res) == n_road, "device-resident and host-buffer paths disagree"

    # max over ranks
    dev_ms, e2e_ms, lean_ms = allreduce_max([dev_ms, e2e_s * 1e3, lean_ms], device="cuda")
    if with_order is not None:
        with_order["dev_ms"], with_order["e2e_ms"] = allreduce_max([with_order["dev_ms"], with_order["e2e_ms"]], device="cuda")
    total_road = allreduce_sum([n_road], device="cuda")[0]

    if rank == 0:
        K = args.steps
        scans = world * B * K
        value = scans / (dev_ms / 1e3)
        e2e = scans / (e2e_ms / 1e3)
        peak, peak_src = hbm_peak()
        dom = max(ktimes, key=ktimes.get)
        dom_ms = ktimes[dom]
        algo_bytes = ALGO_BYTES_PER_POINT * n * B              # per launch: every kernel launch covers the whole batch
        achieved = algo_bytes / (dom_ms / 1e3) / 1e9
        ksum = sum(ktimes.values())
        line = {
            "metric": "scans_per_sec", "value": value, "unit": "scans/s", "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32/f64",
            "data": "synthetic",
            "config": workload_config(args.shape),
            "step": f"a batch of {B} distinct scans per GPU",
            "batch_per_gpu": B, "mpoints_per_sec": value * n / 1e6,
            "l2": f"inputs of one step are {B * n * 16 / 2**20:.0f} MiB per GPU (> 126 MB L2), no reuse between steps",
            "parallelism": f"scan-batch sharding x{world}, no data-path collective",
            "e2e": {"value": e2e, "unit": "scans/s", "h2d_bytes_per_step": B * n * 16,
                    "d2h_bytes_per_step": B * n * 4 + B * C.sizeof(UrfResult), "mpoints_per_sec": e2e * n / 1e6,
                    "pcie": {"h2d_gbs": B * n * 16 / h2d_ms / 1e6, "d2h_gbs": B * n * 4 / d2h_ms / 1e6,
                             "copy_only_ms_per_step": max(h2d_ms, d2h_ms), "both_directions_at_once_ms_per_step": bidir_ms,
                             "note": "the same pinned buffers copied with nothing else going on, rank 0: each direction alone, and both "
                                     "directions at the same time on two streams — the latter is the floor of an e2e step"}},
            "gpu_launches": launches, "road_points_labelled": total_road,
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": ncu_traffic(dom), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": algo_bytes, "kernel_ms": dom_ms,
                         "kernel_share_of_step": ktimes[dom] / ksum,
                         "pipeline_frac": (algo_bytes / (dev_ms / K / 1e3) / 1e9) / peak,
                         "timing": f"CUDA events in front of every kernel on the library's stream, {kprof} single-stream steps "
                                   f"({serial_ms:.3f} ms/step) run inside bench.py right after the timed region, whose {K} steps "
                                   "overlap 2 sub-batches on 2 streams",
                         "kernel_ms_per_step": {k: v for k, v in sorted(ktimes.items(), key=lambda kv: -kv[1])}},
            "clocks": clocks,
        }
        # same scans through urf_process_batch_xyz: 12-byte points in, int8 labels out (13 B per point over PCIe instead of 20)
        line["e2e_lean"] = {"value": scans / (lean_ms / 1e3), "unit": "scans/s", "h2d_bytes_per_step": B * n * 12,
                            "d2h_bytes_per_step": B * n + B * C.sizeof(UrfResult), "entry": "urf_process_batch_xyz (opt-in; e2e above is the float4 / int32 drop-in call)"}
        if with_order is not None:           # labels + vertices + emission order (k_sort_rings inside the timed region)
            line["with_order"] = {"value": scans / (with_order["dev_ms"] / 1e3), "unit": "scans/s", "ms_per_step": with_order["dev_ms"] / K,
                                  "kernel_ms_per_step": with_order.get("kernel_ms"),
                                  "e2e": {"value": scans / (with_order["e2e_ms"] / 1e3), "unit": "scans/s", "h2d_bytes_per_step": B * n * 16,
                                          "d2h_bytes_per_step": 2 * B * n * 4 + B * C.sizeof(UrfResult)}}
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        print(json.dumps(line), flush=True)
    det.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
