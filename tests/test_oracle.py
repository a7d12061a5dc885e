"""The oracle itself: the CPU restatement (oracle/urf_oracle.cpp) is pinned against the golden fixtures generated from the
UNMODIFIED reference (tests/golden/make_golden.py) and against the reference's stored results on seeded random parameter
draws (tests/golden/ref_runs/random_params.npz)."""
import numpy as np
import pytest

from oracle.pyoracle import PortOracle
from urban_road_filter_b200 import FULL_ROI, make_params
from urban_road_filter_b200.api import build_markers
from urban_road_filter_b200.synth import make_scan

from util import Golden, StoredRefRuns, assert_matches_golden, golden_names, random_params_case


@pytest.fixture(scope="module")
def port():
    return PortOracle()


@pytest.mark.parametrize("name", golden_names())
def test_port_matches_reference_golden(port, name):
    g = Golden(name)
    r = port.run(g.cloud, g.params())
    assert_matches_golden(g, r, build_markers)


@pytest.mark.parametrize("seed", range(6))
def test_port_matches_reference_random_params(port, seed):
    """Seeded random draws over the LidarFilters.cfg parameter ranges (cfg/LidarFilters.cfg:10-84)."""
    pts, prm = random_params_case(seed)
    r = StoredRefRuns("random_params").run(str(seed), pts, prm)
    p = port.run(pts, prm)
    assert r.published == (p.status == 0)
    if r.published:
        assert np.array_equal(r.label, p.label)
        if not (p.flags & 4):
            lab = p.label[p.order]
            assert np.array_equal(r.road_ids, p.order[lab == 1])
            assert np.array_equal(r.curb_ids, p.order[lab == 2])


def test_port_edge_cases(port):
    prm = make_params(**FULL_ROI)
    empty = port.run(np.zeros((0, 4), np.float32), prm)
    assert empty.status == 1 and empty.n_roi == 0
    nan = make_scan("C1", 0)[:2000].copy()
    nan[::7, 0] = np.nan
    nan[3::11, 2] = np.inf
    r = port.run(nan, prm)
    assert np.all(r.label[::7] == -1) and np.all(r.label[3::11] == -1)
    allzero = np.zeros((100, 4), np.float32)          # x + y + z == 0 -> dropped by the ROI lambda
    assert port.run(allzero, prm).status == 1
