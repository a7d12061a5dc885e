"""Small scans through the code paths added in round 2, for compute-sanitizer: both marker searches (one CTA per scan /
a grid of CTAs for scans above 300 k points), both ring detectors, the emission-order counting sort and its fallback,
the radius-tie path (restated std::sort by one thread), the registration repair inside k_scan_offsets, the lean and record
entries."""
import sys
sys.path.insert(0, ".")
import numpy as np
from oracle.pyoracle import PortOracle
from urban_road_filter_b200 import api, make_params, FULL_ROI
from urban_road_filter_b200.synth import SHAPES, make_scan, random_cloud

prm = make_params(**FULL_ROI)
pts = make_scan("C1", 3)
det = api.Detector(max_points=30000, max_batch=4, params=prm)
base = det.filtered(pts)
tie = pts.copy(); tie[1000:1300, :3] = tie[3000:3300, :3]                      # equal radii -> std::sort emulation
assert det.filtered(tie).flags & 2
assert det.filtered(random_cloud(5000, 5)).flags & 1                            # speculation refuted -> repair in k_scan_offsets
det.set_params(make_params(curb_points=7, **FULL_ROI)); det.filtered(pts)      # one-position-per-thread detector
det.set_params(prm)
rs = det.filtered_batch_records([np.ascontiguousarray(pts[:, :3]), np.ascontiguousarray(pts[:9000, :3])], 12, 0, 4, 8, -1, want_order=True)
assert np.array_equal(rs[0].label, base.label)
flat = make_scan("C1", 4).copy(); flat[:, 2] = -1.8                              # no edges: every sector refined
det.filtered(flat)
det.close()
# OS1-64 sectors (364 points) are sorted near-first; in a flat / half-flat world the walks run off the prefix:
# k_star_refine (remainder sort behind the prefix + warp-wide resumed walk) on every / every other sector
det = api.Detector(max_points=131072, max_batch=1, params=prm)
big = make_scan("C2", 5)
ref = det.filtered(big)
for variant in ("flat", "half"):
    w = big.copy()
    w[(w[:, 0] < 0) if variant == "half" else slice(None), 2] = -1.8
    a = det.filtered(w)
    det.set_option(4, 0); b = det.filtered(w); det.set_option(4, 1)             # whole-sector sorting: same result
    assert np.array_equal(a.label, b.label) and np.array_equal(a.order, b.order), variant
det.close()
# a scan above 300 k points: the grid marker search (k_markers_grid x 2 + k_verts), against the CPU oracle
sh = SHAPES["C5"]
cut = make_scan("C5", 6)[:320000]
prm5 = make_params(channels=sh.channels, interval=sh.interval, **FULL_ROI)
det = api.Detector(max_points=cut.shape[0], max_batch=1, params=prm5)
r = det.filtered(cut)
o = PortOracle().run(cut, prm5)
assert r.status == o.status == 0 and np.array_equal(r.label, o.label)
assert r.n_vert == o.n_vert and np.array_equal(r.vert, o.vert)
print("ok")
det.close()
