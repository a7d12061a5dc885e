"""Generates tests/golden/*.npz by running the UNMODIFIED reference (oracle/_ref/liburf_ref.so, built from the
reference's sources by `make -C oracle ref REF=<reference checkout>`) on seeded synthetic clouds. Needs the reference
build; the fixtures let the tests compare with the reference wherever it cannot be built.

    python tests/golden/make_golden.py [--only <name prefix>]

Each fixture holds: params (cfg overrides), the input cloud (or, for big clouds, the generator recipe + sha256 of the
bytes it must produce), and what the reference published: per-point labels (recovered from the roi/road/curb clouds),
the road / curb / road_probably clouds as input-index lists in emission order, and the road_marker line strips with
simplification off (exact vertices) and with the cfg defaults.

tests/golden/ref_runs/<family>.npz (name prefix "ref_runs") hold the reference's results on the cases of the tests that
compare with it directly (util.StoredRefRuns): the seeded random parameter draws of tests/test_oracle.py, the marker
strips of tests/test_markers.py and the labels of scripts/fuzz_model.py's first 60 seeds.
"""
from __future__ import annotations

import hashlib
import json
import os
import platform
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from fuzz_model import fuzz_case, fuzz_key, ref_compares, run_ref_isolated  # noqa: E402
from oracle.pyoracle import RefOracle, RefResult  # noqa: E402
from urban_road_filter_b200 import FULL_ROI, make_params  # noqa: E402
from urban_road_filter_b200.synth import SHAPES, make_scan, random_cloud  # noqa: E402
from util import MARKER_EPS, REF_RUNS_DIR, marker_case, random_params_case, ref_run_digest  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

CASES = [
    # name, recipe, store_input, param overrides
    ("c1_full_s0", dict(kind="scan", shape="C1", seed=0, order="column"), True, dict(**FULL_ROI)),
    ("c1_default_ring_s1", dict(kind="scan", shape="C1", seed=1, order="ring"), True, dict()),
    ("c1_full_xonly", dict(kind="scan", shape="C1", seed=0, order="column"), False, dict(z_zero_method=0, star_shaped_method=0, **FULL_ROI)),
    ("c1_full_zonly", dict(kind="scan", shape="C1", seed=0, order="column"), False, dict(x_zero_method=0, star_shaped_method=0, **FULL_ROI)),
    ("c1_full_staronly_beam", dict(kind="scan", shape="C1", seed=0, order="column"), False, dict(x_zero_method=0, z_zero_method=0, starbeam_filter=1, **FULL_ROI)),
    ("c1_full_xdir1_cp3", dict(kind="scan", shape="C1", seed=0, order="column"), False, dict(xDirection=1, curb_points=3, beamZone=45.5, **FULL_ROI)),
    ("c1_full_noblind_cp12", dict(kind="scan", shape="C1", seed=0, order="column"), False, dict(blind_spots=0, curb_points=12, **FULL_ROI)),
    ("random5000_s1_ties", dict(kind="random", n=5000, seed=1), True, dict(**FULL_ROI)),
    ("random5000_s5_specfail", dict(kind="random", n=5000, seed=5), True, dict(**FULL_ROI)),
    ("tiny29", dict(kind="scan", shape="C1", seed=0, order="column", head=29), False, dict(**FULL_ROI)),
    ("c2_default_s0", dict(kind="scan", shape="C2", seed=0, order="column"), False, dict()),
    ("c2_full_ring_s1", dict(kind="scan", shape="C2", seed=1, order="ring"), False, dict(**FULL_ROI)),
    ("c3_full_s0", dict(kind="scan", shape="C3", seed=0, order="column"), False, dict(**FULL_ROI)),
    ("c4_full_s0", dict(kind="scan", shape="C4", seed=0, order="column"), False, dict(channels=128, interval=0.07, **FULL_ROI)),
    # BASELINE config 5 (256 rings x 4096 columns = 1,048,576 points) and its detector ablation. The reference needs 12.9 GB
    # for its channels x N array3D and about 80 s per call here (page faults + its O(n^2) ring sort): run with --only c5
    ("c5_full_s0", dict(kind="scan", shape="C5", seed=0, order="column"), False, dict(channels=256, interval=0.07, **FULL_ROI)),
    ("c5_full_staronly", dict(kind="scan", shape="C5", seed=0, order="column"), False, dict(channels=256, interval=0.07, x_zero_method=0, z_zero_method=0, **FULL_ROI)),
    ("c5_full_xonly", dict(kind="scan", shape="C5", seed=0, order="column"), False, dict(channels=256, interval=0.07, star_shaped_method=0, z_zero_method=0, **FULL_ROI)),
    ("c5_full_zonly", dict(kind="scan", shape="C5", seed=0, order="column"), False, dict(channels=256, interval=0.07, star_shaped_method=0, x_zero_method=0, **FULL_ROI)),
]


def cloud_from_recipe(rc: dict) -> np.ndarray:
    if rc["kind"] == "scan":
        pts = make_scan(rc["shape"], rc["seed"], order=rc["order"])
    else:
        pts = random_cloud(rc["n"], rc["seed"])
    if "head" in rc:
        pts = pts[: rc["head"]].copy()
    return pts


def strips_to_arrays(strips):
    meta = np.array([[s[0], s[1], s[2], len(s[3])] for s in strips], np.int32).reshape(-1, 4)
    pts = np.concatenate([s[3] for s in strips], 0) if strips else np.zeros((0, 3))
    return meta, pts.astype(np.float64)


def ref_run_arrays(key: str, pts, prm, r, fields) -> dict:
    """One case of a ref_runs family: the digest of its inputs, whether the reference crashed, and `fields` of its result."""
    out = {f"{key}.digest": np.array(ref_run_digest(pts, prm)), f"{key}.crashed": np.int8(r is None)}
    for f in fields if r is not None else ():
        if f == "strips":
            out[f"{key}.strips_meta"], out[f"{key}.strips_pts"] = strips_to_arrays(r.strips)
        elif f == "label":
            out[f"{key}.label"] = r.label.astype(np.int8)
        else:
            out[f"{key}.{f}"] = np.asarray(getattr(r, f))
    return out


def make_ref_runs(ref: RefOracle):
    os.makedirs(REF_RUNS_DIR, exist_ok=True)
    runs = {}
    for seed in range(6):
        pts, prm = random_params_case(seed)
        runs.update(ref_run_arrays(str(seed), pts, prm, ref.run(pts, prm), ("published", "label", "road_ids", "curb_ids")))
    np.savez_compressed(os.path.join(REF_RUNS_DIR, "random_params.npz"), **runs)
    runs = {}
    for seed in range(4):
        for k, eps in enumerate(MARKER_EPS):
            pts, prm = marker_case(seed, eps)
            runs.update(ref_run_arrays(f"{seed}_{k}", pts, prm, ref.run(pts, prm, ghostcount=0), ("markers_published", "strips")))
    np.savez_compressed(os.path.join(REF_RUNS_DIR, "markers.npz"), **runs)
    runs = {}
    for seed in range(60):
        _, pts, prm = fuzz_case(seed)
        if ref_compares(pts.shape[0], False):
            label = run_ref_isolated(ref, pts, prm)
            r = None
            if label is not None:
                r = RefResult()
                r.label = label
            runs.update(ref_run_arrays(fuzz_key(seed), pts, prm, r, ("label",)))
    np.savez_compressed(os.path.join(REF_RUNS_DIR, "fuzz.npz"), **runs)
    print(f"ref_runs: {len(runs)} arrays of fuzz cases, sizes " +
          ", ".join(f"{f} {os.path.getsize(os.path.join(REF_RUNS_DIR, f))} B" for f in sorted(os.listdir(REF_RUNS_DIR))))


def main():
    only = sys.argv[sys.argv.index("--only") + 1] if "--only" in sys.argv else ""      # name prefix; default: everything but c5
    ref = RefOracle()
    if "ref_runs".startswith(only):
        make_ref_runs(ref)
    env = dict(machine=platform.machine(), libc=" ".join(platform.libc_ver()), python=platform.python_version(),
               numpy=np.__version__)
    for name, recipe, store, over in CASES:
        if (only and not name.startswith(only)) or (not only and name.startswith("c5")):
            continue
        pts = cloud_from_recipe(recipe)
        sha = hashlib.sha256(pts.tobytes()).hexdigest()
        r0 = ref.run(pts, make_params(simple_poly_allow=0, poly_z_avg_allow=0, **over), ghostcount=0)
        r1 = ref.run(pts, make_params(**over), ghostcount=3)
        assert np.array_equal(r0.label, r1.label)
        m0, p0 = strips_to_arrays(r0.strips)
        m1, p1 = strips_to_arrays(r1.strips)
        out = dict(meta=json.dumps(dict(name=name, recipe=recipe, params=over, sha256=sha, n=int(pts.shape[0]), env=env)),
                   published=np.int32(r0.published), label=r0.label.astype(np.int8), n_roi=np.int32(r0.n_roi),
                   road_ids=r0.road_ids, curb_ids=r0.curb_ids, prob_ids=r0.prob_ids,
                   strips_raw_meta=m0, strips_raw_pts=p0, strips_cfg_meta=m1, strips_cfg_pts=p1,
                   markers_published=np.int32(r0.markers_published), ghost_after=np.int32(r1.ghostcount))
        if store:
            out["cloud"] = pts
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
        print(f"{name:28s} n={pts.shape[0]:7d} published={r0.published} roi={r0.n_roi} road={r0.n_road} curb={r0.n_curb} "
              f"strips={len(r0.strips)} sha={sha[:12]}")


if __name__ == "__main__":
    main()
