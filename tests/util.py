"""Shared helpers of the test-suite: golden fixtures, comparisons, the CPU model binding."""
from __future__ import annotations

import ctypes as C
import glob
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle.pyoracle import OracleDebug, RefResult  # noqa: E402
from urban_road_filter_b200 import FULL_ROI, UrfParams, UrfResult, make_params  # noqa: E402
from urban_road_filter_b200.ctypes_abi import URF_MAX_CHANNELS, URF_MAX_VERTS  # noqa: E402
from urban_road_filter_b200.synth import make_scan, random_cloud  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
REF_RUNS_DIR = os.path.join(GOLDEN_DIR, "ref_runs")
VERT_TOL = 1e-4     # metres: BASELINE.json north_star tolerance for curb-polyline vertices


_SCAN_CACHE: dict = {}


def cached_scan(shape, seed, order):
    """make_scan with a one-entry cache per (shape, seed, order): the four C5 fixtures share one 1M-point cloud."""
    key = (shape, seed, order)
    if key not in _SCAN_CACHE:
        if len(_SCAN_CACHE) > 3:
            _SCAN_CACHE.clear()
        _SCAN_CACHE[key] = make_scan(shape, seed, order=order)
    return _SCAN_CACHE[key]


def golden_names() -> list[str]:
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))


class Golden:
    def __init__(self, name: str):
        z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
        self.meta = json.loads(str(z["meta"]))
        self.name = name
        self.params_over = self.meta["params"]
        rc = self.meta["recipe"]
        if "cloud" in z.files:
            self.cloud = z["cloud"]
        else:
            self.cloud = cached_scan(rc["shape"], rc["seed"], rc["order"]) if rc["kind"] == "scan" else random_cloud(rc["n"], rc["seed"])
            if "head" in rc:
                self.cloud = self.cloud[: rc["head"]].copy()
        sha = hashlib.sha256(np.ascontiguousarray(self.cloud).tobytes()).hexdigest()
        assert sha == self.meta["sha256"], f"{name}: the synthetic generator no longer reproduces the fixture's input cloud"
        self.published = bool(z["published"])
        self.label = z["label"].astype(np.int32)
        self.road_ids, self.curb_ids, self.prob_ids = z["road_ids"], z["curb_ids"], z["prob_ids"]
        self.strips_raw = self._strips(z["strips_raw_meta"], z["strips_raw_pts"])
        self.strips_cfg = self._strips(z["strips_cfg_meta"], z["strips_cfg_pts"])
        self.markers_published = bool(z["markers_published"])
        self.ghost_after = int(z["ghost_after"])

    @staticmethod
    def _strips(meta, pts):
        out, k = [], 0
        for sid, act, red, cnt in meta:
            out.append((int(sid), int(act), int(red), pts[k: k + cnt]))
            k += cnt
        return out

    def params(self, **extra) -> UrfParams:
        return make_params(**{**self.params_over, **extra})


def assert_matches_golden(g: Golden, res, build_markers, check_order: bool = True):
    """res: anything with status/label/order/ring_start/n_rings/vert (PortResult, ScanResult, model result)."""
    if not g.published:
        assert res.status == 1, "reference published nothing (piece < 30)"
        return
    assert res.status == 0
    assert np.array_equal(res.label, g.label), f"{g.name}: labels differ at {np.nonzero(res.label != g.label)[0][:10]}"
    ties = bool(res.flags & 4)
    if check_order and res.order is not None and not ties:
        lab = res.label[res.order]
        assert np.array_equal(res.order[lab == 1], g.road_ids), "road cloud emission order"
        assert np.array_equal(res.order[lab == 2], g.curb_ids), "curb cloud emission order"
        prob = res.order[res.ring_start[10]: res.ring_start[11]] if res.n_rings > 10 else np.zeros(0, np.int32)
        assert np.array_equal(prob, g.prob_ids), "road_probably cloud"
    if ties:
        return   # reference order of equal azimuths comes from its unstable quicksort; vertices may legitimately differ
    # vertices, through the marker tail with simplification off: exact (x, y, z) of every strip point
    strips, _ = build_markers(g.params(simple_poly_allow=0, poly_z_avg_allow=0), res.vert, 0)
    compare_strips(strips, g.strips_raw, g.name + " raw strips")
    strips, ghost = build_markers(g.params(), res.vert, 3)
    compare_strips(strips, g.strips_cfg, g.name + " cfg strips")
    if g.markers_published:
        assert ghost == g.ghost_after


def compare_strips(mine, ref, what):
    assert len(mine) == len(ref), f"{what}: {len(mine)} strips vs {len(ref)}"
    for a, b in zip(mine, ref):
        assert a[0] == b[0] and a[1] == b[1], f"{what}: id/action {a[:3]} vs {b[:3]}"
        if a[1] == 2:
            continue      # DELETE markers carry no geometry
        assert a[2] == b[2], f"{what}: colour"
        assert a[3].shape == b[3].shape, f"{what}: strip {a[0]} has {a[3].shape[0]} points, reference {b[3].shape[0]}"
        assert np.all(np.abs(a[3] - b[3]) <= VERT_TOL), f"{what}: vertex off by {np.abs(a[3] - b[3]).max()} m"


def random_params_case(seed: int):
    """(cloud, parameters) of seeded random draw `seed` over the LidarFilters.cfg parameter ranges (cfg/LidarFilters.cfg:10-84)."""
    rng = np.random.default_rng(100 + seed)
    pts = make_scan("C1", 10 + seed, order=("column", "ring")[seed % 2]) if seed % 3 else random_cloud(6000, seed, rings=12)
    prm = make_params(
        x_zero_method=int(rng.integers(0, 2)), z_zero_method=int(rng.integers(0, 2)), star_shaped_method=int(rng.integers(0, 2)),
        blind_spots=int(rng.integers(0, 2)), xDirection=int(rng.integers(0, 3)), interval=float(rng.uniform(0.05, 0.5)),
        curb_height=float(rng.uniform(0.01, 0.2)), curb_points=int(rng.integers(1, 12)), beamZone=float(rng.uniform(10, 100)),
        cylinder_deg_x=float(rng.uniform(90, 180)), cylinder_deg_z=float(rng.uniform(90, 180)),
        curb_slope_deg=float(rng.uniform(10, 90)), kdev_param=float(rng.uniform(0.5, 5)), kdist_param=float(rng.uniform(0.4, 10)),
        starbeam_filter=int(rng.integers(0, 2)), dmin_param=int(rng.integers(3, 30)),
        **(FULL_ROI if seed % 2 else dict(min_x=-20.0, max_x=40.0, min_y=-15.0, max_y=15.0, min_z=-3.0, max_z=1.0)))
    return pts, prm


MARKER_EPS = (0.05, 0.7, 3.0)


def marker_case(seed: int, eps: float):
    """(cloud, parameters) of a whole VLP-16 scan whose road_marker strips are simplified with tolerance `eps`."""
    return make_scan("C1", 20 + seed), make_params(poly_s_param=eps, **FULL_ROI)


def ref_run_digest(pts: np.ndarray, prm: UrfParams) -> str:
    """sha256 of a cloud's bytes and of every parameter value: names the inputs a stored reference run was made on."""
    h = hashlib.sha256(np.ascontiguousarray(pts, np.float32).tobytes())
    h.update(repr([getattr(prm, f) for f, _ in UrfParams._fields_]).encode())
    return h.hexdigest()


class StoredRefRuns:
    """What the unmodified reference (oracle.pyoracle.RefOracle.run) returned on named cases, recorded by
    tests/golden/make_golden.py into tests/golden/ref_runs/<family>.npz, so that comparisons with the reference also run
    where it cannot be built. Each case holds the digest of its inputs and the fields its tests compare."""

    def __init__(self, family: str):
        z = np.load(os.path.join(REF_RUNS_DIR, family + ".npz"))
        self._cases: dict[str, dict] = {}
        for f in z.files:
            key, field = f.rsplit(".", 1)
            self._cases.setdefault(key, {})[field] = z[f]

    def __contains__(self, key: str) -> bool:
        return key in self._cases

    def __len__(self) -> int:
        return len(self._cases)

    def run(self, key: str, pts: np.ndarray, prm: UrfParams):
        """The stored RefOracle().run(pts, prm) of case `key`, or None where the reference crashed on it."""
        a = self._cases[key]
        assert str(a["digest"]) == ref_run_digest(pts, prm), f"{key}: not the cloud and parameters the reference was run on"
        if a["crashed"]:
            return None
        r = RefResult()
        for f, v in a.items():
            if f in ("published", "markers_published"):
                setattr(r, f, bool(v))
            elif f == "label":
                r.label = v.astype(np.int32)
            elif f not in ("digest", "crashed", "strips_meta", "strips_pts"):
                setattr(r, f, v)
        if "strips_meta" in a:
            r.strips = Golden._strips(a["strips_meta"], a["strips_pts"])
        return r


def feq(a: np.ndarray, b: np.ndarray) -> bool:
    """bitwise float equality, any NaN == any NaN (x86 and the GPU produce different NaN bit patterns for 0/0)"""
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    a = np.where(np.isnan(a), np.float32(np.nan), a)
    b = np.where(np.isnan(b), np.float32(np.nan), b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


class ModelResult:
    pass


class CpuModel:
    """build/libmodel.so: the kernels' logic functions run sequentially on the CPU (tests/kat/model_check.cpp)."""

    def __init__(self):
        self.lib = C.CDLL(os.path.join(ROOT, "build", "libmodel.so"))
        self.lib.urf_model_run.restype = C.c_int
        self.lib.urf_model_run.argtypes = [C.c_void_p, C.c_int, C.POINTER(UrfParams), C.POINTER(UrfResult),
                                           C.POINTER(OracleDebug), C.c_int]

    def run(self, pts, prm, force_exact=0) -> ModelResult:
        pts = np.ascontiguousarray(pts, np.float32)
        n, m = pts.shape[0], max(pts.shape[0], 1)
        res = UrfResult()
        a = dict(label=np.full(m, -1, np.int32), ring=np.full(m, -1, np.int32), order=np.zeros(m, np.int32),
                 ring_start=np.zeros(URF_MAX_CHANNELS + 1, np.int32))
        for k, v in a.items():
            setattr(res, k, v.ctypes.data_as(C.POINTER(C.c_int32)))
        d = dict(alpha_v=np.full(m, np.nan, np.float32), az=np.full(m, np.nan, np.float32), d2=np.full(m, np.nan, np.float32),
                 star_mark=np.zeros(m, np.int8), det_label=np.full(m, -1, np.int8),
                 ring_angle=np.full(URF_MAX_CHANNELS, np.nan, np.float32), max_dist=np.full(URF_MAX_CHANNELS, np.nan, np.float32))
        dbg = OracleDebug(**{k: v.ctypes.data for k, v in d.items()})
        rc = self.lib.urf_model_run(pts.ctypes.data, n, C.byref(prm), C.byref(res), C.byref(dbg), force_exact)
        assert rc == 0, rc
        r = ModelResult()
        r.__dict__.update(a)
        r.__dict__.update(d)
        for f in ("status", "n_roi", "n_rings", "n_order", "n_road", "n_curb", "n_vert", "flags"):
            setattr(r, f, int(getattr(res, f)))
        r.label, r.ring, r.order = r.label[:n], r.ring[:n], r.order[: res.n_order]
        r.vert = np.ctypeslib.as_array(res.vert).reshape(URF_MAX_VERTS, 4)[: res.n_vert].copy()
        return r


def stage_diffs(o, m, n: int, check_order: bool = True) -> list[str]:
    """Names of the stages in which result m (model / GPU) differs from the oracle's debug run o."""
    bad = []
    if o.status != m.status:
        return ["status"]
    if o.status != 0:
        return bad
    for f in ("alpha_v", "az", "d2"):
        if getattr(m, f, None) is not None and not feq(getattr(o, f)[:n], getattr(m, f)[:n]):
            bad.append(f)
    for f in ("star_mark", "det_label"):
        if getattr(m, f, None) is not None and not np.array_equal(getattr(o, f)[:n], getattr(m, f)[:n]):
            bad.append(f)
    if o.n_rings != m.n_rings:
        bad.append("n_rings")
    elif getattr(m, "ring_angle", None) is not None:
        if not feq(o.ring_angle[: o.n_rings], m.ring_angle[: o.n_rings]):
            bad.append("ring_angle")
        if not feq(o.max_dist[: o.n_rings], m.max_dist[: o.n_rings]):
            bad.append("max_dist")
    if m.ring is not None and not np.array_equal(o.ring, m.ring):
        bad.append("ring")
    if not np.array_equal(o.label, m.label):
        bad.append("label")
    if (o.n_roi, o.n_road, o.n_curb, o.n_order) != (m.n_roi, m.n_road, m.n_curb, m.n_order):
        bad.append("counts")
    if (o.flags & 2) != (m.flags & 2):
        bad.append("sector_tie_flag")
    ties = bool(o.flags & 4)
    if check_order and m.order is not None:
        if bool(m.flags & 4) != ties:
            bad.append("azimuth_tie_flag")
        if not ties and not np.array_equal(o.order, m.order):
            bad.append("order")
        if not np.array_equal(o.ring_start[: o.n_rings + 1], m.ring_start[: o.n_rings + 1]):
            bad.append("ring_start")
    if not ties and (o.n_vert != m.n_vert or not feq(o.vert, m.vert)):
        bad.append("vert")
    return bad
