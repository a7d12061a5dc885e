"""Marker tail (urf_build_markers, lidar_segmentation.cpp:369-602): the Douglas-Peucker step. Boost.Geometry is not part of the
reference tree, so `simplify` is PARITY UNPINNED (DESIGN.md): the product states the published algorithm iteratively
(urban_road_filter_b200/csrc/urf_markers.cpp), the reference build of the oracle states it recursively
(oracle/shim/boost/geometry.hpp). These tests pin both to the algorithm's defining properties and to each other."""
import numpy as np
import pytest

from oracle.pyoracle import PortOracle
from urban_road_filter_b200 import api, make_params

from util import MARKER_EPS, StoredRefRuns, marker_case


def strip_points(vert_xy, eps, simplify=True):
    """One green strip through urf_build_markers; returns its (x, y) points."""
    n = len(vert_xy)
    v = np.zeros((n, 4), np.float32)
    v[:, :2] = vert_xy
    v[:, 2] = -1.8
    prm = make_params(simple_poly_allow=int(simplify), poly_s_param=eps, poly_z_avg_allow=0)
    strips, _ = api.build_markers(prm, v, 0)
    assert len(strips) == 1 and strips[0][1] == 0 and strips[0][2] == 0
    return strips[0][3][:, :2].astype(np.float32)


def dist_to_polyline(p, poly):
    a, b = poly[:-1].astype(np.float64), poly[1:].astype(np.float64)
    v, w = b - a, p.astype(np.float64) - a
    t = np.clip((w * v).sum(1) / np.maximum((v * v).sum(1), 1e-30), 0, 1)
    return np.sqrt((((a + t[:, None] * v) - p) ** 2).sum(1)).min()


def wiggly(n, seed):
    rng = np.random.default_rng(seed)
    x = np.cumsum(rng.uniform(0.2, 1.0, n))
    y = np.cumsum(rng.normal(0, 0.3, n)) + 2.0 * np.sin(x / 3.0)
    return np.stack([x, y], 1).astype(np.float32)


@pytest.mark.parametrize("seed", range(8))
def test_simplify_properties(seed):
    pts = wiggly(40 + 37 * seed, seed)
    prev = None
    for eps in (0.0, 0.05, 0.2, 0.7, 2.0, 10.0, 1e6):
        out = strip_points(pts, eps)
        # a subsequence of the input, end points kept
        idx = []
        j = 0
        for q in out:
            while not np.array_equal(pts[j], q):
                j += 1
            idx.append(j)
            j += 1
        assert idx[0] == 0 and idx[-1] == len(pts) - 1
        # every dropped point lies within eps of the simplified line (the Douglas-Peucker guarantee)
        for k in range(len(pts)):
            if k not in idx:
                assert dist_to_polyline(pts[k], out) <= eps * (1 + 1e-5) + 1e-6
        # nested in eps: what survives a larger tolerance survives every smaller one
        if prev is not None:
            assert set(idx) <= prev
        prev = set(idx)
    assert len(strip_points(pts, 1e6)) == 2
    assert np.array_equal(strip_points(pts, 0.7, simplify=False), pts)


def test_simplify_collinear_and_degenerate():
    line = np.stack([np.arange(50, dtype=np.float32), 0.5 * np.arange(50, dtype=np.float32)], 1)
    assert len(strip_points(line, 0.01)) == 2                       # exactly collinear: only the end points survive
    spike = line.copy()
    spike[25, 1] += 3.0
    out = strip_points(spike, 0.7)
    assert len(out) == 5 and np.array_equal(out[2], spike[25])      # the spike and its two flanks survive
    three = np.array([[0, 0], [1, 5], [2, 0]], np.float32)
    assert len(strip_points(three, 0.7)) == 3 and len(strip_points(three, 6.0)) == 2
    dup = np.array([[0, 0], [0, 0], [0, 0], [4, 0]], np.float32)   # repeated points / zero-length chord
    assert np.array_equal(strip_points(dup, 0.1), dup[[0, 3]])
    closed = np.array([[0, 0], [3, 4], [0, 0]], np.float32)        # chord of length 0: distance to the point itself
    assert len(strip_points(closed, 0.7)) == 3


@pytest.mark.parametrize("seed", range(4))
def test_iterative_and_recursive_statements_agree(seed):
    """The product (iterative) against the reference build, whose marker tail (the unmodified lidar_segmentation.cpp:369-602)
    calls the shim's recursive statement: same strips for the same candidate vertices, at several tolerances. The
    reference's strips are stored in tests/golden/ref_runs/markers.npz."""
    stored = StoredRefRuns("markers")
    for k, eps in enumerate(MARKER_EPS):
        pts, prm = marker_case(seed, eps)
        r = stored.run(f"{seed}_{k}", pts, prm)
        if not r.markers_published:
            continue
        o = PortOracle().run(pts, prm)
        mine, _ = api.build_markers(prm, o.vert, 0)
        assert len(mine) == len(r.strips)
        for a, b in zip(mine, r.strips):
            assert a[:3] == b[:3] and a[3].shape == b[3].shape and np.allclose(a[3], b[3], atol=1e-6)
