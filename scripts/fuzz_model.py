#!/usr/bin/env python
"""CPU fuzz of the kernels' arithmetic and stage logic: the CPU model (tests/kat/model_check.cpp — the same
urf_logic.cuh functions the kernels call, in the kernels' stage order) against the oracle port and against the unmodified
reference, on seeded random parameter draws over the LidarFilters.cfg ranges and varied clouds (sensor layouts, flat
worlds, quantised ranges = equal radii, random clouds). No GPU needed. The reference's labels come from
tests/golden/ref_runs/fuzz.npz (recorded by tests/golden/make_golden.py) for the seeds stored there, and from the
reference build (oracle/_ref) for other seeds where that exists.
usage: fuzz_model.py [first_seed] [count] [big]   -> one line per mismatch, a summary line at the end
("big": whole OS1-64 / HDL-64E / OS2-128 scans instead of the small clouds, a few tenths of a second per case and side)"""
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

from oracle.pyoracle import PortOracle, RefOracle  # noqa: E402
from urban_road_filter_b200 import FULL_ROI, make_params  # noqa: E402
from urban_road_filter_b200.synth import make_scan, random_cloud  # noqa: E402
from util import CpuModel, StoredRefRuns, stage_diffs  # noqa: E402


def fuzz_case(seed: int, big: bool = False):
    """(kind, cloud, parameters) of one fuzz case."""
    rng = np.random.default_rng(9000 + seed)
    kind = seed % 6
    ch, iv = 64, None
    if big:
        shape = ("C2", "C2", "C3", "C4")[seed % 4]
        pts = make_scan(shape, 100 + seed, order="ring" if seed % 4 == 1 else "column")
        if shape == "C4":
            ch, iv = 128, 0.07
        if seed % 5 == 0:
            pts[:, 2] = np.where(pts[:, 0] < rng.uniform(-30, 30), -1.8, pts[:, 2])        # partly flat world
    elif kind == 0:
        pts = make_scan("C1", 100 + seed, order="column")
    elif kind == 1:
        pts = make_scan("C1", 100 + seed, order="ring")
        pts[:, 2] = np.where(pts[:, 0] < rng.uniform(-30, 30), -1.8, pts[:, 2])            # partly flat world
    elif kind == 2:
        pts = random_cloud(int(rng.integers(2000, 12000)), seed, rings=int(rng.integers(4, 40)))
    elif kind == 3:
        pts = make_scan("C1", 100 + seed, order="column")                                  # quantised ranges: equal radii in a sector
        q = float(rng.choice([0.002, 0.01, 0.05]))
        r = np.sqrt((pts[:, :3].astype(np.float64) ** 2).sum(1))
        rq = np.maximum(np.round(r / q), 1) * q
        pts[:, :3] = (pts[:, :3] * (rq / np.maximum(r, 1e-9))[:, None]).astype(np.float32)
    elif kind == 4:
        pts = make_scan("C2", 100 + seed, order="column")[:: int(rng.integers(2, 5))].copy()   # thinned OS1-64
    else:
        pts = make_scan("C4", 100 + seed, order="ring")[::4].copy(); ch, iv = 128, 0.07
    prm = make_params(
        x_zero_method=int(rng.integers(0, 2)), z_zero_method=int(rng.integers(0, 2)), star_shaped_method=int(rng.integers(0, 2)),
        blind_spots=int(rng.integers(0, 2)), xDirection=int(rng.integers(0, 3)),
        interval=float(iv if iv is not None else rng.uniform(0.05, 0.5)),
        curb_height=float(rng.uniform(0.01, 0.2)), curb_points=int(rng.choice([5, 5, 3, 9, 17, 1, 30])), beamZone=float(rng.uniform(10, 100)),
        cylinder_deg_x=float(rng.uniform(90, 180)), cylinder_deg_z=float(rng.uniform(90, 180)),
        curb_slope_deg=float(rng.uniform(10, 90)), kdev_param=float(rng.uniform(0.5, 5)), kdist_param=float(rng.uniform(0.4, 10)),
        starbeam_filter=int(rng.integers(0, 2)), dmin_param=int(rng.integers(3, 30)), channels=ch,
        **(FULL_ROI if seed % 2 else dict(min_x=-20.0, max_x=40.0, min_y=-15.0, max_y=15.0, min_z=-3.0, max_z=1.0)))
    return kind, pts, prm


def fuzz_key(seed: int, big: bool = False) -> str:
    return f"{'big' if big else 'small'}_{seed}"


def ref_compares(n: int, big: bool) -> bool:
    """Which cases are also run through the reference (it allocates channels x N x 48 B per scan)."""
    return n <= 40000 or big


def run_ref_isolated(ref, pts, prm):
    """The reference's labels, computed in a forked child: it has undefined behaviour of its own on some inputs
    (SURVEY.md H5) and a crash there must not end the sweep. Returns None when the child crashed."""
    fd, tmp = tempfile.mkstemp(suffix=".npy")
    os.close(fd)
    try:
        pid = os.fork()
        if pid == 0:
            try:
                np.save(tmp, np.asarray(ref.run(pts, prm, ghostcount=0).label, np.int32))
                os._exit(0)
            except BaseException:
                os._exit(3)
        _, status = os.waitpid(pid, 0)
        return np.load(tmp) if status == 0 else None
    finally:
        os.remove(tmp)


def main():
    first = int(sys.argv[1]) if len(sys.argv) > 1 else 0
    count = int(sys.argv[2]) if len(sys.argv) > 2 else 50
    big = len(sys.argv) > 3 and sys.argv[3] == "big"
    port, model = PortOracle(), CpuModel()
    stored = StoredRefRuns("fuzz")
    ref = RefOracle() if RefOracle.available() else None
    bad = nref = nties = ncrash = 0
    road = curb = 0
    t0 = time.time()
    for seed in range(first, first + count):
        kind, pts, prm = fuzz_case(seed, big)
        n = pts.shape[0]
        o = port.run(pts, prm, debug=True)
        m = model.run(pts, prm, 0)
        d = stage_diffs(o, m, n)
        if d:
            bad += 1
            print(f"seed {seed} kind {kind}: model vs port: {d[:3]}", flush=True)
        nties += bool(m.flags & 2)
        road += int((np.asarray(m.label) == 1).sum()); curb += int((np.asarray(m.label) == 2).sum())
        if not ref_compares(n, big):
            continue
        key = fuzz_key(seed, big)
        if key in stored:
            r = stored.run(key, pts, prm)
            rl = None if r is None else r.label
        elif ref is not None:
            rl = run_ref_isolated(ref, pts, prm)
        else:
            continue
        if rl is None:
            ncrash += 1
            print(f"seed {seed} kind {kind}: the reference itself crashed", flush=True)
            continue
        nref += 1
        if not np.array_equal(rl, np.asarray(m.label)):
            bad += 1
            print(f"seed {seed} kind {kind}: model vs REFERENCE labels differ at {int((rl != np.asarray(m.label)).sum())} points (flags {m.flags})", flush=True)
    print(f"fuzz_model: seeds {first}..{first + count - 1}: {count} cases vs the port, {nref} of them also vs the unmodified reference, "
          f"{ncrash} reference crashes, {nties} with equal radii in a sector, {road} road / {curb} curb labels; mismatching cases {bad}; {time.time() - t0:.0f} s")


if __name__ == "__main__":
    main()
