"""CPU model of the CUDA pipeline (tests/kat/model_check.cpp): the SAME logic functions the kernels call
(urban_road_filter_b200/csrc/urf_logic.cuh) run sequentially on the host, diffed stage by stage against the oracle.
This pins the reformulated stages (speculative registration + verification, blindSpots window tables, marker aggregates)
without a GPU; tests/test_gpu_parity.py then checks the kernels' plumbing around the same functions."""
import itertools

import numpy as np
import pytest

from oracle.pyoracle import PortOracle
from urban_road_filter_b200 import FULL_ROI, make_params
from urban_road_filter_b200.api import build_markers
from urban_road_filter_b200.synth import SHAPES, make_scan, random_cloud

from util import CpuModel, Golden, StoredRefRuns, assert_matches_golden, golden_names, stage_diffs


@pytest.fixture(scope="module")
def both():
    return PortOracle(), CpuModel()


def _check(both, pts, prm, force_exact=0):
    port, model = both
    o = port.run(pts, prm, debug=True)
    m = model.run(pts, prm, force_exact)
    assert stage_diffs(o, m, pts.shape[0]) == []
    return m


@pytest.mark.parametrize("name", [n for n in golden_names() if not n.startswith(("c3", "c4", "c5"))])
def test_model_matches_golden(name):
    g = Golden(name)
    assert_matches_golden(g, CpuModel().run(g.cloud, g.params()), build_markers)


@pytest.mark.parametrize("cfg,seed,roi,order", [("C1", 0, "def", "column"), ("C1", 1, "full", "ring"), ("C2", 2, "full", "column"),
                                                 ("C2", 3, "def", "ring"), ("C3", 4, "full", "column")])
def test_model_shapes(both, cfg, seed, roi, order):
    sh = SHAPES[cfg]
    _check(both, make_scan(cfg, seed, order=order), make_params(channels=sh.channels, interval=sh.interval, **(FULL_ROI if roi == "full" else {})))


def test_model_detector_toggles(both):
    pts = make_scan("C1", 3)
    for xz, zz, st, bs in itertools.product((0, 1), repeat=4):
        _check(both, pts, make_params(x_zero_method=xz, z_zero_method=zz, star_shaped_method=st, blind_spots=bs, **FULL_ROI))


@pytest.mark.parametrize("kw", [dict(xDirection=1), dict(xDirection=2, starbeam_filter=1), dict(curb_points=1), dict(curb_points=30),
                                dict(beamZone=10), dict(beamZone=45.5), dict(beamZone=100), dict(beamZone=359.5), dict(beamZone=360),
                                dict(curb_height=0.2), dict(curb_slope_deg=5), dict(kdev_param=0.5, kdist_param=10, dmin_param=3),
                                dict(interval=0.05), dict(interval=3.0), dict(channels=11), dict(channels=3), dict(channels=1)])
def test_model_param_sweep(both, kw):
    _check(both, make_scan("C1", 3), make_params(**kw, **FULL_ROI))


@pytest.mark.parametrize("seed", range(6))
def test_model_random_clouds_and_exact_registration(both, seed):
    pts = random_cloud(5000, seed)
    m = _check(both, pts, make_params(**FULL_ROI))
    e = _check(both, pts, make_params(**FULL_ROI), force_exact=1)
    assert e.flags & 1
    assert np.array_equal(m.label, e.label)
    _check(both, random_cloud(20000, seed, rings=40), make_params())


def test_model_speculation_failure_is_repaired(both):
    """random cloud seed 5 defeats the 'first point per elevation bin' speculation; verification must catch it."""
    m = _check(both, random_cloud(5000, 5), make_params(**FULL_ROI))
    assert m.flags & 32 and m.flags & 1


def test_model_zero_elevation_quirk(both):
    """A point straight below the sensor has elevation angle exactly 0: the reference's `angle[j] == 0` sentinel then hides
    that and all later registered angles from the scan (lidar_segmentation.cpp:176)."""
    pts = make_scan("C1", 2)[:6000].copy()
    pts[5] = (1e-5, 2e-5, -1.5, 1.0)       # |z| / d rounds to exactly 1.0f -> acosf -> 0.0, but r and azimuth stay regular
    pts[900] = (3e-5, -1e-5, -1.7, 1.0)
    m = _check(both, pts, make_params(**FULL_ROI))
    assert m.flags & 16 and m.flags & 1


def test_model_fuzz_short():
    """A short run of scripts/fuzz_model.py (random parameter draws x varied clouds; model vs port, and vs the unmodified
    reference's labels stored for these seeds). The long run (3000 cases, 0 mismatches) is recorded in DESIGN.md §2."""
    import os
    import re
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "scripts", "fuzz_model.py"), "0", "60"], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "mismatching cases 0;" in out.stdout, out.stdout[-2000:]
    m = re.search(r"(\d+) of them also vs the unmodified reference, (\d+) reference crashes", out.stdout)
    assert m and int(m.group(1)) > 0 and int(m.group(1)) + int(m.group(2)) == len(StoredRefRuns("fuzz")), out.stdout[-2000:]
