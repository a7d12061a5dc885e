"""Parity tests proper: the CUDA path, called through the C-ABI (urban_road_filter_b200.api.Detector -> liburf_b200.so),
against the CPU oracle on the same seeded inputs and against the golden fixtures generated from the unmodified reference.
Bar: per-point labels, ring ids, emission order bit-exact; marker vertices within 1e-4 m (they are in fact bit-exact)."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle.pyoracle import PortOracle
from urban_road_filter_b200 import FULL_ROI, make_params
from urban_road_filter_b200 import api
from urban_road_filter_b200.ctypes_abi import URF_ERR_INVALID
from urban_road_filter_b200.synth import SHAPES, make_scan, random_cloud

from util import Golden, assert_matches_golden, golden_names, stage_diffs

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def det():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    d = api.Detector(max_points=300_000, max_batch=8)
    yield d
    d.close()


@pytest.fixture(scope="module")
def port():
    return PortOracle()


class GpuDebug:
    """Stage intermediates of scan 0 of the last call, re-indexed by input index like the oracle's debug run."""

    def __init__(self, det, res, n):
        N = res.n_order
        self.__dict__.update(res.__dict__ if hasattr(res, "__dict__") else {s: getattr(res, s) for s in res.__slots__})
        a = det.debug_fetch(0, 0, np.float32, n)
        self.alpha_v = np.where(a < 0, np.nan, a).astype(np.float32)
        ring = det.debug_fetch(0, 2, np.int16, n)
        in_ring = ring >= 0
        self.az = np.where(in_ring, det.debug_fetch(0, 4, np.float32, n), np.float32(np.nan)).astype(np.float32)
        self.d2 = np.where(in_ring, det.debug_fetch(0, 5, np.float32, n), np.float32(np.nan)).astype(np.float32)
        self.star_mark = None      # the device keeps one mark for all three detectors
        self.det_label = np.where(in_ring, det.debug_fetch(0, 1, np.uint8, n).astype(np.int8), np.int8(-1)).astype(np.int8)
        self.ring_angle = None


def check(det, port, pts, prm, exact=False):
    det.set_params(prm)
    det.set_option(0, 1 if exact else 0)
    r = det.filtered(pts)
    det.set_option(0, 0)
    o = port.run(pts, prm, debug=True)
    if o.status == 0 and r.status == 0:
        g = GpuDebug(det, r, pts.shape[0])
        bad = stage_diffs(o, g, pts.shape[0])
    else:
        bad = [] if o.status == r.status else ["status"]
    assert bad == [], f"stages differing from the oracle: {bad}"
    return r


@pytest.fixture(scope="module")
def det_big():
    """A detector sized for BASELINE config 5 (1,048,576 points), created on first use."""
    holder = {}

    def get():
        if "d" not in holder:
            holder["d"] = api.Detector(max_points=1_048_576, max_batch=1)
        return holder["d"]

    yield get
    if "d" in holder:
        holder["d"].close()


@pytest.mark.parametrize("name", golden_names())
def test_gpu_matches_reference_golden(det, det_big, name):
    """Fixtures produced by the UNMODIFIED reference (tests/golden/make_golden.py), C1 .. C5 shapes: C5 = 256 rings x 4096
    columns with `channels` = 256, all detectors and one detector at a time."""
    g = Golden(name)
    d = det if g.cloud.shape[0] <= det.max_points else det_big()
    d.set_params(g.params())
    assert_matches_golden(g, d.filtered(g.cloud), api.build_markers)


@pytest.mark.parametrize("cfg,seed,roi,order", [("C1", 0, "def", "column"), ("C1", 1, "full", "ring"), ("C2", 2, "full", "column"),
                                                 ("C2", 3, "def", "ring"), ("C3", 4, "full", "column"), ("C4", 5, "full", "ring")])
def test_gpu_shapes(det, port, cfg, seed, roi, order):
    sh = SHAPES[cfg]
    check(det, port, make_scan(cfg, seed, order=order), make_params(channels=sh.channels, interval=sh.interval, **(FULL_ROI if roi == "full" else {})))


@pytest.mark.parametrize("mask", range(16))
def test_gpu_detector_toggles(det, port, mask):
    check(det, port, make_scan("C1", 3), make_params(x_zero_method=mask & 1, z_zero_method=(mask >> 1) & 1,
                                                      star_shaped_method=(mask >> 2) & 1, blind_spots=(mask >> 3) & 1, **FULL_ROI))


@pytest.mark.parametrize("kw", [dict(xDirection=1), dict(xDirection=2, starbeam_filter=1), dict(curb_points=1), dict(curb_points=30),
                                dict(beamZone=10), dict(beamZone=45.5), dict(beamZone=100), dict(beamZone=360),
                                dict(curb_height=0.2), dict(curb_slope_deg=5), dict(kdev_param=0.5, kdist_param=10, dmin_param=3),
                                dict(interval=0.05), dict(interval=3.0), dict(channels=11), dict(channels=3), dict(channels=1)])
def test_gpu_param_sweep(det, port, kw):
    check(det, port, make_scan("C1", 3), make_params(**kw, **FULL_ROI))


@pytest.mark.parametrize("seed", range(10))
def test_gpu_random_parameter_draws(det, port, seed):
    """Seeded random draws over the LidarFilters.cfg parameter ranges (cfg/LidarFilters.cfg:10-84), alternating sensor
    layouts, ROI presets and cloud kinds: every stage against the oracle."""
    rng = np.random.default_rng(500 + seed)
    kind = seed % 4
    if kind == 0:
        pts, ch, iv = make_scan("C1", 30 + seed, order="column"), 64, None
    elif kind == 1:
        pts, ch, iv = make_scan("C2", 30 + seed, order="ring"), 64, None
    elif kind == 2:
        pts, ch, iv = random_cloud(8000, seed, rings=14), 64, None
    else:
        pts, ch, iv = make_scan("C4", 30 + seed, order="column"), 128, 0.07
    prm = make_params(
        x_zero_method=int(rng.integers(0, 2)), z_zero_method=int(rng.integers(0, 2)), star_shaped_method=int(rng.integers(0, 2)),
        blind_spots=int(rng.integers(0, 2)), xDirection=int(rng.integers(0, 3)),
        interval=float(iv if iv is not None else rng.uniform(0.05, 0.5)),
        curb_height=float(rng.uniform(0.01, 0.2)), curb_points=int(rng.choice([5, 5, 3, 9, 17])), beamZone=float(rng.uniform(10, 100)),
        cylinder_deg_x=float(rng.uniform(90, 180)), cylinder_deg_z=float(rng.uniform(90, 180)),
        curb_slope_deg=float(rng.uniform(10, 90)), kdev_param=float(rng.uniform(0.5, 5)), kdist_param=float(rng.uniform(0.4, 10)),
        starbeam_filter=int(rng.integers(0, 2)), dmin_param=int(rng.integers(3, 30)), channels=ch,
        **(FULL_ROI if seed % 2 else dict(min_x=-20.0, max_x=40.0, min_y=-15.0, max_y=15.0, min_z=-3.0, max_z=1.0)))
    check(det, port, pts, prm)


@pytest.mark.parametrize("seed", range(6))
def test_gpu_random_clouds_and_exact_registration(det, port, seed):
    pts = random_cloud(5000, seed)
    a = check(det, port, pts, make_params(**FULL_ROI))
    b = check(det, port, pts, make_params(**FULL_ROI), exact=True)
    assert b.flags & 1
    assert np.array_equal(a.label, b.label)
    check(det, port, random_cloud(20000, seed, rings=40), make_params())


def test_gpu_speculation_failure_is_repaired(det, port):
    r = check(det, port, random_cloud(5000, 5), make_params(**FULL_ROI))
    assert r.flags & 1        # exact registration ran after the failed verification


def test_gpu_zero_elevation_quirk(det, port):
    pts = make_scan("C1", 2)[:6000].copy()
    pts[5] = (1e-5, 2e-5, -1.5, 1.0)
    pts[900] = (3e-5, -1e-5, -1.7, 1.0)
    r = check(det, port, pts, make_params(**FULL_ROI))
    assert r.flags & 1


def test_gpu_nan_azimuth_is_flagged(det, port):
    """A ROI point with x == y == 0 has azimuth NaN: the documented deviation (it belongs to no blindSpots window or marker
    bin) is reported in urf_result.flags bit3; a scan without such a point does not carry the bit."""
    pts = make_scan("C1", 6).copy()
    prm = make_params(**FULL_ROI)
    det.set_params(prm)
    assert not (det.filtered(pts).flags & 8)
    pts[1234, :3] = (0.0, 0.0, -1.7)
    r = det.filtered(pts)
    assert r.flags & 8
    o = port.run(pts, prm)                                    # the CPU restatement follows the same policy
    assert np.array_equal(r.label, o.label)


def test_gpu_edge_cases(det, port):
    prm = make_params(**FULL_ROI)
    det.set_params(prm)
    r = det.filtered(np.zeros((0, 4), np.float32))
    assert r.status == 1 and r.n_roi == 0
    r = det.filtered(make_scan("C1", 0)[:29])
    assert r.status == 1 and np.all(r.label == -1)
    nan = make_scan("C1", 0)[:2000].copy()
    nan[::7, 0] = np.nan
    nan[3::11, 2] = np.inf
    check(det, port, nan, prm)
    check(det, port, make_scan("C1", 0), make_params(min_x=100, max_x=101))      # empty ROI
    with pytest.raises(api.UrfError):
        det.filtered(np.zeros((400_000, 4), np.float32))                         # larger than the ctx capacity


def test_gpu_profile_option_after_graphed_call(port):
    """urf_set_option(1, ...) after a CUDA-graph replay: the graph handle is dropped and rebuilt, nothing is destroyed twice
    (the documented flow filtered -> set_option(1, n) -> kernel_times -> set_option(1, 0) -> filtered -> close)."""
    d = api.Detector(max_points=30_000, max_batch=2)
    try:
        prm = make_params(**FULL_ROI)
        d.set_params(prm)
        pts = make_scan("C1", 12)
        o = port.run(pts, prm)
        assert np.array_equal(d.filtered(pts).label, o.label)          # captures the graph
        d.set_option(1, 2)
        assert np.array_equal(d.filtered(pts).label, o.label)          # per-kernel events, no graph
        names = [k for k, _ in d.kernel_times(0)]
        assert any(k.startswith("k_ring_detect") for k in names) and "k_label" in names
        d.set_option(1, 0)
        d.set_option(1, 0)
        assert np.array_equal(d.filtered(pts).label, o.label)          # graph captured again
        d.set_option(1, 1)
    finally:
        d.close()


def test_gpu_batch_equals_single(det, port):
    """Ragged batch: every scan of a batch gets the result it gets alone (scans are independent units)."""
    clouds = [make_scan("C1", 1), make_scan("C2", 2, order="ring"), random_cloud(5000, 5), make_scan("C1", 4)[:29],
              make_scan("C3", 3), np.zeros((0, 4), np.float32), make_scan("C1", 7)[:12345]]
    prm = make_params(**FULL_ROI)
    det.set_params(prm)
    rs = det.filtered_batch(clouds)
    for c, r in zip(clouds, rs):
        o = port.run(c, prm)
        assert o.status == r.status
        if o.status == 0:
            assert stage_diffs(o, r, c.shape[0]) == []


def test_gpu_device_resident_entry_point(det, port):
    """urf_process_batch_device: inputs and labels stay in device memory (what bench.py times as `value`)."""
    prm = make_params(**FULL_ROI)
    det.set_params(prm)
    clouds = [make_scan("C2", s) for s in range(3)]
    S = 131072
    x = torch.zeros((3, S, 4), dtype=torch.float32, device="cuda")
    for b, c in enumerate(clouds):
        x[b, : c.shape[0]] = torch.from_numpy(c).cuda()
    lab = torch.full((3, S), -7, dtype=torch.int32, device="cuda")
    n = (C.c_int * 3)(*[c.shape[0] for c in clouds])
    from urban_road_filter_b200 import UrfResult
    outs = (UrfResult * 3)()
    torch.cuda.synchronize()
    rc = det.lib.urf_process_batch_device(det._ctx, x.data_ptr(), S, n, 3, lab.data_ptr(), outs)
    assert rc == 0
    assert det.last_launch_count() >= 10 and det.last_device_ms() > 0
    host = lab.cpu().numpy()
    for b, c in enumerate(clouds):
        o = port.run(c, prm)
        assert np.array_equal(host[b, : c.shape[0]], o.label)
        assert (outs[b].n_road, outs[b].n_curb, outs[b].n_vert) == (o.n_road, o.n_curb, o.n_vert)


def test_gpu_full_size_c5_and_properties(port):
    """BASELINE config 5 (256 rings x 4096 columns = 1,048,576 points), every detector ablation, vs the oracle; plus
    size-independent properties: idempotence (same cloud twice -> same labels) and batch-order independence."""
    sh = SHAPES["C5"]
    pts = make_scan("C5", 0)
    d = api.Detector(max_points=pts.shape[0], max_batch=2)
    try:
        for kw in (dict(), dict(x_zero_method=0, z_zero_method=0), dict(star_shaped_method=0, z_zero_method=0), dict(star_shaped_method=0, x_zero_method=0)):
            prm = make_params(channels=sh.channels, interval=sh.interval, **kw, **FULL_ROI)
            d.set_params(prm)
            r = d.filtered(pts)
            o = port.run(pts, prm)
            assert stage_diffs(o, r, pts.shape[0]) == []
        a, b = d.filtered_batch([pts, pts[::-1].copy()])
        again = d.filtered(pts)
        assert np.array_equal(a.label, again.label) and np.array_equal(a.vert, again.vert)
        assert a.n_roi == b.n_roi
    finally:
        d.close()


def test_gpu_pipelined_host_batch(port):
    """Batches of 16+ scans go through the chunked three-stream pipeline (H2D / kernels / D2H overlap): same results."""
    d = api.Detector(max_points=30_000, max_batch=24)
    try:
        prm = make_params(**FULL_ROI)
        d.set_params(prm)
        clouds = [make_scan("C1", 40 + s, order=("column", "ring")[s % 2])[: 28800 - 997 * (s % 5)] for s in range(21)]
        clouds[7] = clouds[7][:20]                      # fewer than 30 ROI points: nothing published for this one
        clouds[13] = random_cloud(5000, 5)              # speculation failure inside a chunk
        rs = d.filtered_batch(clouds)
        for c, r in zip(clouds, rs):
            o = port.run(c, prm)
            assert o.status == r.status
            if o.status == 0:
                assert stage_diffs(o, r, c.shape[0]) == []
    finally:
        d.close()


def _model():
    from util import CpuModel
    return CpuModel()


def test_gpu_fallback_paths_big_sector_big_ring_large_cp(det, port):
    """Rarely taken code paths: a star sector with > 8192 points (global-memory bitonic fallback), a ring with ~60k points
    (emission-order sort beyond shared memory), curb_points beyond the shared-memory halo of k_ring_detect."""
    rng = np.random.default_rng(7)
    n = 60000
    az = np.deg2rad(rng.uniform(10.02, 10.98, n))                 # one star sector, one elevation -> one ring
    t = np.sort(rng.uniform(2.0, 50.0, n))[rng.permutation(n)]
    e = np.deg2rad(-12.0)
    pts = np.zeros((n, 4), np.float32)
    pts[:, 0] = t * np.cos(e) * np.cos(az); pts[:, 1] = t * np.cos(e) * np.sin(az); pts[:, 2] = t * np.sin(e) + rng.normal(0, 0.02, n)
    from urban_road_filter_b200.synth import _detie_radius
    _detie_radius(pts, 7)
    check(det, port, pts, make_params(interval=3.0, **FULL_ROI))
    check(det, port, make_scan("C1", 5), make_params(curb_points=40, **FULL_ROI))
    check(det, port, make_scan("C2", 6, order="ring"), make_params(curb_points=33, beamZone=12.5, **FULL_ROI))


def _one_ring_cloud(az_deg, seed):
    rng = np.random.default_rng(seed)
    n = len(az_deg)
    az = np.deg2rad(np.asarray(az_deg, np.float64))
    t = rng.uniform(2.0, 50.0, n)
    e = np.deg2rad(-12.0)
    pts = np.zeros((n, 4), np.float32)
    pts[:, 0] = t * np.cos(e) * np.cos(az); pts[:, 1] = t * np.cos(e) * np.sin(az); pts[:, 2] = t * np.sin(e) + rng.normal(0, 0.02, n)
    from urban_road_filter_b200.synth import _detie_radius
    _detie_radius(pts, seed)
    return pts


def test_gpu_ring_sort_paths(det, port):
    """k_sort_rings: counting sort over azimuth bins (rings up to 4096 points) and its fallbacks — a ring whose points
    crowd into one bin, a ring confined to a two-degree arc (bins adapt to the ring's azimuth range), a ring beyond 4096
    points — all against the oracle's emission order."""
    rng = np.random.default_rng(13)                                  # a seed whose clouds have no exact azimuth ties
    prm = make_params(interval=3.0, **FULL_ROI)
    crowded = rng.permutation(np.concatenate([rng.uniform(100.0, 100.08, 60), rng.uniform(0.0, 359.0, 1940)]))
    arc = rng.uniform(100.0, 130.0, 1200)
    r = check(det, port, _one_ring_cloud(crowded, 1), prm)           # 60 points inside one of the 4096 bins: fallback
    assert r.n_rings == 1 and r.n_order == 2000 and not (r.flags & 4)
    r = check(det, port, _one_ring_cloud(arc, 2), prm)
    assert not (r.flags & 4)
    check(det, port, _one_ring_cloud(rng.uniform(0.0, 359.9, 4096), 3), prm)
    check(det, port, _one_ring_cloud(rng.uniform(0.0, 359.9, 4097), 4), prm)
    check(det, port, _one_ring_cloud(np.sort(rng.uniform(0.0, 359.9, 2048))[::-1], 5), prm)      # descending: the reference's O(n^2) case


def test_gpu_radius_ties_take_the_reference_order(det, port):
    """Exact radius ties inside a sector: the reference's order is what libstdc++'s introsort leaves (std::sort by radius
    alone on the sector's points in push_back order); the tie path reproduces it (urf_stdsort.cuh), so labels — which do
    depend on that order — equal the oracle's, whose star search calls the real std::sort. Flagged in urf_result.flags bit1."""
    for seed, dup in ((8, 400), (9, 40), (10, 1500)):
        pts = make_scan("C1", seed).copy()
        pts[1000:1000 + dup, :3] = pts[3000:3000 + dup, :3]          # exact duplicates -> same sector, same radius
        pts[5000:5200, 2] += 0.3                                      # and height steps among them: the tie order decides labels
        prm = make_params(**FULL_ROI)
        det.set_params(prm)
        r = det.filtered(pts)
        o = port.run(pts, prm)
        m = _model().run(pts, prm)
        assert r.flags & 2 and m.flags & 2 and o.flags & 2
        assert np.array_equal(m.label, o.label), "CPU model of the tie path vs the oracle"
        assert np.array_equal(r.label, o.label) and np.array_equal(r.ring, o.ring)
        if not (r.flags & 4):
            assert np.array_equal(r.order, o.order) and np.array_equal(r.vert, o.vert)
    # quantised ranges (what a real sensor delivers): a flat ring returns the same range in neighbouring columns
    pts = make_scan("C2", 12).copy()
    rng = np.linalg.norm(pts[:, :3], axis=1, keepdims=True)
    q = np.round(rng * 500.0) / 500.0                                 # 2 mm range quantisation along the beam
    pts[:, :3] = (pts[:, :3] / np.maximum(rng, 1e-9) * q).astype(np.float32)
    prm = make_params(**FULL_ROI)
    det.set_params(prm)
    r = det.filtered(pts)
    o = port.run(pts, prm)
    assert np.array_equal(r.label, o.label) and (r.flags & 2) == (o.flags & 2)


def test_gpu_device_resident_multi_stream_groups(port):
    """A device-resident batch of >= 8 scans is spread over four compute streams (offset buffer views, fork/join on the
    context's stream): every scan must still get exactly the oracle's labels, with a ragged batch and a stride larger
    than any scan."""
    d = api.Detector(max_points=30_000, max_batch=20)
    try:
        prm = make_params(**FULL_ROI)
        d.set_params(prm)
        clouds = [make_scan("C1", 60 + s, order=("column", "ring")[s % 2])[: 28800 - 1013 * (s % 4)] for s in range(19)]
        clouds[11] = random_cloud(5000, 5)
        S = 29_696
        x = torch.zeros((19, S, 4), dtype=torch.float32, device="cuda")
        for b, c in enumerate(clouds):
            x[b, : c.shape[0]] = torch.from_numpy(c).cuda()
        lab = torch.full((19, S), -7, dtype=torch.int32, device="cuda")
        n = (C.c_int * 19)(*[c.shape[0] for c in clouds])
        from urban_road_filter_b200 import UrfResult
        outs = (UrfResult * 19)()
        torch.cuda.synchronize()
        for groups in (4, 1):
            d.set_option(2, groups)
            lab.fill_(-7)
            assert d.lib.urf_process_batch_device(d._ctx, x.data_ptr(), S, n, 19, lab.data_ptr(), outs) == 0
            host = lab.cpu().numpy()
            for b, c in enumerate(clouds):
                o = port.run(c, prm)
                assert np.array_equal(host[b, : c.shape[0]], o.label), (groups, b)
                assert np.all(host[b, c.shape[0]:] == -7)            # nothing written beyond the scan
                assert (outs[b].n_road, outs[b].n_curb, outs[b].n_vert, outs[b].n_rings) == (o.n_road, o.n_curb, o.n_vert, o.n_rings)
                assert np.array_equal(np.ctypeslib.as_array(outs[b].vert).reshape(-1, 4)[: o.n_vert], o.vert)
    finally:
        d.close()


@pytest.mark.parametrize("step,ox,oy,oz", [(16, 0, 4, 8), (32, 0, 4, 8), (48, 0, 4, 8), (22, 0, 4, 8), (22, 8, 4, 12), (64, 40, 12, 28)])
def test_gpu_pointcloud2_unpack_on_device(det, port, step, ox, oy, oz):
    """urf_process_cloud2: raw PointCloud2 records (Ouster 48 B, Velodyne 22/32 B incl. records that are not 4-byte aligned,
    shuffled field offsets) unpacked on the device give the same result as the repacked float4 cloud."""
    pts = make_scan("C1", 9)
    n = pts.shape[0]
    raw = np.random.default_rng(step).integers(0, 256, n * step, dtype=np.uint8)      # garbage in the other fields
    rec = raw.reshape(n, step)
    for k, off in enumerate((ox, oy, oz)):
        rec[:, off: off + 4] = pts[:, k: k + 1].copy().view(np.uint8)
    prm = make_params(**FULL_ROI)
    det.set_params(prm)
    r = det.filtered_cloud2(raw, n, step, ox, oy, oz)
    o = port.run(pts, prm)
    assert stage_diffs(o, r, n) == []


def test_gpu_lean_and_batched_record_entries(port):
    """urf_process_batch_xyz (12-byte points in, int8 labels out) and urf_process_cloud2_batch (raw PointCloud2 records of a
    whole batch unpacked on the device), ragged batches large enough for the chunked copy/compute pipeline: labels, order
    and vertices equal the oracle's on the float4 clouds."""
    d = api.Detector(max_points=30_000, max_batch=20)
    try:
        prm = make_params(**FULL_ROI)
        d.set_params(prm)
        clouds = [make_scan("C1", 80 + s, order=("column", "ring")[s % 2])[: 28800 - 911 * (s % 5)] for s in range(18)]
        clouds[5] = clouds[5][:17]
        clouds[9] = random_cloud(5000, 5)
        exp = [port.run(c, prm) for c in clouds]
        xyz = [np.ascontiguousarray(c[:, :3]) for c in clouds]
        for label8 in (True, False):
            rs = d.filtered_batch_records(xyz, 12, 0, 4, 8, -1, want_order=True, label8=label8)
            for o, r, c in zip(exp, rs, clouds):
                assert o.status == r.status
                if o.status == 0:
                    r.ring = None
                    assert stage_diffs(o, r, c.shape[0]) == []
                else:
                    assert np.all(r.label == -1)
        recs = [_cloud2_records(c, 22, 0, 4, 8, 12, seed=i).reshape(-1) for i, c in enumerate(clouds)]     # Velodyne-like, unaligned
        rs = d.filtered_batch_records(recs, 22, 0, 4, 8, 12, want_order=True, label8=True)
        for o, r, c in zip(exp, rs, clouds):
            assert o.status == r.status
            if o.status == 0:
                r.ring = None
                assert stage_diffs(o, r, c.shape[0]) == []
        one = d.filtered_batch_records(recs[:3], 22, 0, 4, 8, 12, want_order=True, label8=False)              # small batch: one chunk
        for o, r, c in zip(exp[:3], one, clouds[:3]):
            r.ring = None
            assert stage_diffs(o, r, c.shape[0]) == []
    finally:
        d.close()


def _cloud2_records(pts, step, ox, oy, oz, oi, seed=0):
    n = pts.shape[0]
    rec = np.random.default_rng(seed).integers(0, 256, (n, step), dtype=np.uint8)     # garbage in the other fields
    for k, off in enumerate((ox, oy, oz, oi)):
        if off >= 0:
            rec[:, off: off + 4] = pts[:, k: k + 1].copy().view(np.uint8)
    return rec.reshape(-1)


def _expect_records(pts, ids, with_intensity=True):
    e = np.zeros((len(ids), 8), np.float32)
    e[:, 0:3] = pts[ids, 0:3]
    e[:, 3] = 1.0
    if with_intensity:
        e[:, 4] = pts[ids, 3]
    return e


@pytest.mark.parametrize("name", golden_names())
def test_gpu_packed_clouds_match_reference_goldens(det, name):
    """urf_process_cloud2_packed (SURVEY.md §8 f1): the four clouds packed on the device are, record for record and in
    order, the clouds the UNMODIFIED reference published for the same input (fixtures of tests/golden)."""
    g = Golden(name)
    pts = g.cloud
    n = pts.shape[0]
    if n > det.max_points:
        pytest.skip("larger than the module's detector")
    det.set_params(g.params())
    raw = _cloud2_records(pts, 48, 0, 4, 8, 16, seed=n)                 # Ouster-like 48-byte records, intensity at 16
    r, cl = det.filtered_cloud2_packed(raw, n, 48, 0, 4, 8, 16, want_labels=True)
    if not g.published:
        assert r.status == 1 and all(len(v) == 0 for v in cl.values())
        return
    assert r.status == 0
    np.testing.assert_array_equal(r.label, g.label)
    for key, ids in (("road", g.road_ids), ("curb", g.curb_ids), ("road_probably", g.prob_ids), ("roi", np.flatnonzero(g.label >= 0))):
        exp = _expect_records(pts, np.asarray(ids, np.int64))
        assert cl[key].shape == exp.shape, f"{key}: {cl[key].shape[0]} records, reference published {exp.shape[0]}"
        assert cl[key].tobytes() == exp.tobytes(), f"{key}: packed cloud differs from the reference's"


@pytest.mark.parametrize("shape,step,offs", [("C1", 22, (0, 4, 8, 12)), ("C2", 32, (0, 4, 8, 16)), ("C2", 64, (40, 12, 28, -1))])
def test_gpu_packed_clouds_match_oracle(det, port, shape, step, offs):
    """Packed clouds against the oracle's labels + emission order on larger scans, default and full ROI, with records
    that are not 4-byte aligned and without an intensity field."""
    pts = make_scan(shape, 21)
    n = pts.shape[0]
    for prm in (make_params(), make_params(**FULL_ROI)):
        det.set_params(prm)
        raw = _cloud2_records(pts, step, *offs, seed=step)
        r, cl = det.filtered_cloud2_packed(raw, n, step, *offs)
        o = port.run(pts, prm)
        assert r.status == o.status == 0
        lab = np.asarray(o.label)
        order = np.asarray(o.order[: o.n_order])
        rs = np.asarray(o.ring_start)
        wi = offs[3] >= 0
        exp = {"road": order[lab[order] == 1], "curb": order[lab[order] == 2], "roi": np.flatnonzero(lab >= 0),
               "road_probably": order[rs[10]: rs[11]] if len(rs) > 11 else order[:0]}
        for key, ids in exp.items():
            e = _expect_records(pts, ids, wi)
            assert cl[key].shape == e.shape and cl[key].tobytes() == e.tobytes(), key
        assert r.label is None and (r.n_road, r.n_curb) == (len(exp["road"]), len(exp["curb"]))


@pytest.mark.parametrize("variant", ["scan", "flat", "half_flat"])
@pytest.mark.parametrize("shape", ["C1", "C2", "C3", "C4"])
def test_gpu_near_first_star_sort(det, port, shape, variant):
    """k_star_sort_warp sorts only the points below a sampled pivot radius and k_star_scan redoes (tab.refine) the sectors
    whose edge search runs off that prefix. A flat world has no edge at all (every sector is refined), a half-flat one
    mixes both paths; each must give the oracle's result, and the same result as whole-sector sorting (option 4 = 0).
    Typical star sectors: about 80 points (C1: below the near-first threshold), 380 (C2, C3) and 760 (C4: whole-sector
    sorts of more than 512 points go to k_star_sort_big)."""
    sh = SHAPES[shape]
    pts = make_scan(shape, 31)
    if variant == "flat":
        pts[:, 2] = -1.8
    elif variant == "half_flat":
        pts[pts[:, 0] < 0, 2] = -1.8
    n = pts.shape[0]
    prm = make_params(channels=sh.channels, interval=sh.interval, **FULL_ROI)
    det.set_params(prm)
    o = port.run(pts, prm, debug=True)
    if variant == "flat":
        assert int((np.asarray(o.star_mark) == 2).sum()) == 0
    res = {}
    for mode in (1, 0):
        det.set_option(4, mode)
        r = det.filtered(pts)
        assert stage_diffs(o, GpuDebug(det, r, n), n) == [], f"star_prefix={mode}"
        res[mode] = r
    det.set_option(4, 1)
    np.testing.assert_array_equal(res[0].label, res[1].label)
    np.testing.assert_array_equal(res[0].vert, res[1].vert)


# options 5-12 selected tuning variants that were removed: each accepts only the value now built in
RETIRED_OPTIONS = {5: 0, 6: 0, 7: 0, 8: 46, 9: 1, 10: 17, 11: 1, 12: 16}


def test_gpu_retired_options(det):
    """A retired option set to its built-in value is accepted, so old tuning command lines keep working; asking for a
    removed variant is refused with URF_ERR_INVALID instead of silently running the built-in one."""
    for opt, builtin in RETIRED_OPTIONS.items():
        det.set_option(opt, builtin)
    removed = ((5, 4), (6, 1), (7, 1), (8, 4), (8, 8), (9, 0), (9, 2), (10, 14), (11, 0), (12, 32))
    for opt, value in removed:
        with pytest.raises(api.UrfError) as e:
            det.set_option(opt, value)
        assert e.value.code == URF_ERR_INVALID, (opt, value)
