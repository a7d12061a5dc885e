// tests/kat/model_check.cpp — CPU model of the CUDA pipeline (TEST CODE, not a product path and not a fallback).
//
// Runs the SAME host+device logic functions the kernels call (urban_road_filter_b200/csrc/urf_logic.cuh, compiled for the
// host with -ffp-contract=off), stage by stage in the order of the kernel pipeline, with sequential stand-ins for what
// the GPU does with atomics, stable partitions and sorts. tests/test_model.py diffs its outputs against the oracle, so
// the reformulated stages (speculative ring registration + verification, blindSpots as window tables, marker search as
// order-independent aggregates) are checked on the CPU before any GPU run. Entry point has the oracle's signature.
#include <algorithm>
#include <cstring>
#include <vector>

#include "../../urban_road_filter_b200/csrc/urf_logic.cuh"
#include "../../urban_road_filter_b200/csrc/urf_stdsort.cuh"
#include "../../urban_road_filter_b200/csrc/urf_host.hpp"

using namespace urf;

struct urf_oracle_debug {   // same layout as oracle/urf_oracle.cpp
  float* alpha_v; float* az; float* d2; int8_t* star_mark; int8_t* det_label; float* ring_angle; float* max_dist;
};

namespace {

// exact registration, mirrors register_exact_cta (sequential form of the rounds)
int register_exact(const std::vector<float>& alpha, float interval, int channels, std::vector<float>& reg, std::vector<int>& idx) {
  std::vector<float> vis;
  bool frozen = false;
  int i_last = -1;
  const int n = (int)alpha.size();
  while ((int)reg.size() < channels) {
    int istar = -1;
    for (int i = i_last + 1; i < n; i++) {
      const float a = alpha[i];
      if (a < 0.0f) continue;
      bool cov = false;
      for (float v : vis) if (fabsf(URF_FSUB(v, a)) <= interval) { cov = true; break; }
      if (!cov) { istar = i; break; }
    }
    if (istar < 0) break;
    const float a = alpha[istar];
    reg.push_back(a); idx.push_back(istar);
    if (!frozen) { if (a == 0.0f) frozen = true; else vis.push_back(a); }
    i_last = istar;
  }
  return (int)reg.size();
}

}  // namespace

extern "C" int urf_model_run(const float* xyzi, int n, const urf_params* up, urf_result* out, const urf_oracle_debug* dbg,
                             int force_exact) {
  if (validate_params(up) != URF_OK) return URF_ERR_INVALID;
  static float beam_d[kSectKeys], beam_o[kSectKeys], Kfi;
  static unsigned char beam_yx[kSectKeys];
  static bool init = false;
  if (!init) { host_beam_init(beam_d, beam_o, beam_yx, &Kfi); init = true; }
  DevParams prm;
  narrow_params(up, &prm, Kfi, force_exact, 1);
  std::vector<float> newY;
  host_newY(newY, n);

  out->status = URF_OK; out->n_in = n; out->n_roi = 0; out->n_rings = 0; out->n_order = 0; out->n_road = 0;
  out->n_curb = 0; out->n_vert = 0; out->flags = 0; out->reserved = 0;
  if (out->label) for (int i = 0; i < n; i++) out->label[i] = URF_LABEL_OUTSIDE;
  if (out->ring) for (int i = 0; i < n; i++) out->ring[i] = -1;
  int flags = 0;

  // ---- k_points
  std::vector<float> alpha(n, -1.0f), az(n, 0.f), d2(n, 0.f);      // az / d2: input order, ROI points only
  std::vector<unsigned> firstidx(kElevBins + 1, 0xffffffffu);
  int n_roi = 0;
  for (int i = 0; i < n; i++) {
    const float x = xyzi[4 * i], y = xyzi[4 * i + 1], z = xyzi[4 * i + 2];
    if (!roi_keep(prm, x, y, z)) continue;
    n_roi++;
    float a;
    point_angles(x, y, z, &a, &d2[i], &az[i]);
    {                                      // the shared-squares form must agree with the two separate reference expressions
      float d_ref, az_ref;
      planar_az(x, y, &d_ref, &az_ref);
      if (fbits(a) != fbits(elev_alpha(x, y, z)) || fbits(d_ref) != fbits(d2[i]) || fbits(az_ref) != fbits(az[i])) return -101;
    }
    alpha[i] = a;
    const int bin = elev_bin(a);
    if (firstidx[bin] > (unsigned)i) firstidx[bin] = (unsigned)i;
    if (a == 0.0f) flags |= F_ZERO_ALPHA;
    if (az[i] != az[i]) flags |= F_NAN_AZIMUTH;
  }
  out->n_roi = n_roi;
  if (n_roi < 30) { out->status = URF_TOO_FEW_POINTS; return 0; }

  // ---- k_register
  std::vector<float> reg; std::vector<int> ridx;
  bool exact = prm.force_exact || (flags & F_ZERO_ALPHA);
  if (!exact) {
    std::vector<unsigned> cand;
    for (unsigned v : firstidx) if (v != 0xffffffffu) cand.push_back(v);
    if ((int)cand.size() > kMaxCand) exact = true;
    else {
      std::sort(cand.begin(), cand.end());
      for (unsigned c : cand) {
        if ((int)reg.size() >= prm.channels) break;
        const float a = alpha[c];
        bool cov = false;
        for (float v : reg) if (fabsf(URF_FSUB(v, a)) <= prm.interval) cov = true;
        if (!cov) { reg.push_back(a); ridx.push_back((int)c); }
      }
    }
  }
  if (exact) { reg.clear(); ridx.clear(); register_exact(alpha, prm.interval, prm.channels, reg, ridx); flags |= F_EXACT_REG; }

  ScanTab* tabp = new ScanTab();
  ScanTab& tab = *tabp;
  std::vector<short> ringid(n, -1), sect(n, -1);
  int R = 0;
  auto publish = [&]() {
    R = (int)reg.size();
    std::vector<std::pair<float, int>> pr(R);
    for (int t = 0; t < R; t++) pr[t] = {reg[t], ridx[t]};
    std::sort(pr.begin(), pr.end());
    for (int t = 0; t < kRingKeys; t++) { tab.angle[t] = 0.f; tab.regidx[t] = 0x7fffffff; tab.regorder[t] = 0x7fffffff; }
    for (int t = 0; t < R; t++) { tab.angle[t] = pr[t].first; tab.regidx[t] = pr[t].second; tab.regorder[t] = ridx[t]; }
  };
  publish();
  // ---- k_assign (+ verify, + repair)
  std::vector<unsigned short> lut(kElevBins + 1);
  auto assign_all = [&](bool verify) {
    bool viol = false;
    for (int e = 0; e <= kElevBins; e++) lut[e] = (unsigned short)ring_lut_entry(tab.angle, R, prm.interval, e);
    for (int i = 0; i < n; i++) {
      const float a = alpha[i];
      ringid[i] = -1; sect[i] = -1;
      if (a < 0.0f) continue;
      int lo, lo_ref;
      ringid[i] = (short)assign_ring_from(tab.angle, R, a, prm.interval, lut[elev_bin(a)], &lo);
      if (ringid[i] != assign_ring(tab.angle, R, a, prm.interval, &lo_ref) || lo != lo_ref) return true;   // LUT search != binary search: report as violation (tests fail)
      if (verify && registration_violation(tab.angle, tab.regidx, tab.regorder, R, prm.channels, prm.interval, a, i, lo)) viol = true;
      if (prm.star) sect[i] = (short)star_sector(prm, xyzi[4 * i], xyzi[4 * i + 1], beam_d, beam_o, beam_yx);
    }
    return viol;
  };
  if (assign_all(!(flags & F_EXACT_REG))) {
    flags |= F_SPEC_VIOLATION | F_EXACT_REG;
    reg.clear(); ridx.clear();
    register_exact(alpha, prm.interval, prm.channels, reg, ridx);
    publish();
    assign_all(false);
  }
  // ---- k_scan_offsets + k_scatter (stable partitions)
  std::vector<int> ring_start(kRingKeys + 1, 0), sect_start(kSectKeys + 1, 0);
  for (int i = 0; i < n; i++) { if (ringid[i] >= 0) ring_start[ringid[i] + 1]++; if (sect[i] >= 0) sect_start[sect[i] + 1]++; }
  for (int k = 0; k < kRingKeys; k++) ring_start[k + 1] += ring_start[k];
  for (int k = 0; k < kSectKeys; k++) sect_start[k + 1] += sect_start[k];
  const int N = ring_start[kRingKeys];
  std::vector<float4> bpt(std::max(N, 1)), spt(std::max(sect_start[kSectKeys], 1));
  {
    std::vector<int> rr(ring_start.begin(), ring_start.end() - 1), ss(sect_start.begin(), sect_start.end() - 1);
    for (int i = 0; i < n; i++) {
      const float x = xyzi[4 * i], y = xyzi[4 * i + 1], z = xyzi[4 * i + 2];
      if (ringid[i] >= 0) bpt[rr[ringid[i]]++] = make_float4(x, y, z, URF_I2F(i));
      if (sect[i] >= 0) spt[ss[sect[i]]++] = make_float4(star_radius(x, y), z, URF_I2F(i), 0.f);
    }
  }

  // ---- k_star_sort + k_star_scan
  std::vector<unsigned char> mark(n, 0);
  if (prm.star) {
    for (int s = 0; s < kSectKeys; s++) {
      const int base = sect_start[s], m = sect_start[s + 1] - base;
      if (m <= 0) continue;
      // the GPU sorts a sector by (radius bits, input index); when that meets equal radii it puts the points back into
      // input (= push_back) order and runs the restated std::sort (urf_stdsort.cuh) — the reference's own tie order
      std::vector<urfsort::El> keys(m);
      for (int t = 0; t < m; t++) keys[t] = ((unsigned long long)fbits(spt[base + t].x) << 32) | (unsigned)URF_F2I(spt[base + t].z);
      std::sort(keys.begin(), keys.end());
      bool tie = false;
      for (int t = 1; t < m; t++) if ((unsigned)(keys[t - 1] >> 32) == (unsigned)(keys[t] >> 32)) tie = true;
      if (tie) {
        flags |= F_TIE_SECTOR;
        std::sort(keys.begin(), keys.end(), [](urfsort::El a, urfsort::El b) { return (unsigned)a < (unsigned)b; });   // by input index
        urfsort::std_sort(keys.data(), m);
      }
      std::vector<float4> sorted(m);
      for (int t = 0; t < m; t++) {
        const int idx = (int)(unsigned)keys[t];
        sorted[t] = make_float4(bitsf((unsigned)(keys[t] >> 32)), xyzi[4 * idx + 2], URF_I2F(idx), 0.f);
      }
      const int hit = star_scan_sector(prm, sorted.data(), m);
      if (hit >= 0) mark[URF_F2I(sorted[hit].z)] = 2;
    }
  }

  // ---- k_star_scan's curb_hit + k_ring_detect
  const size_t nb = (size_t)prm.channels * kDegBins;
  std::vector<unsigned> cmin(nb, 0x7f800000u), cmax(nb, 0u);
  std::vector<unsigned short> ne((size_t)prm.channels * (kDegBins + 1), 0);
  auto curb_hit = [&](int idx, int k) {
    mark[idx] = 2;
    if (k < 0) k = ringid[idx];
    if (k < 0) return;
    const float a = az[idx];
    if (a >= 0.0f) {
      const size_t o = (size_t)k * kDegBins + deg_bin(a);
      if (fbits(a) < cmin[o]) cmin[o] = fbits(a);
      if (fbits(a) > cmax[o]) cmax[o] = fbits(a);
    }
  };
  std::vector<unsigned char> star_mark(mark);           // the star search alone (debug output)
  for (int i = 0; i < n; i++) if (star_mark[i] == 2) curb_hit(i, -1);
  for (int k = 0; k < kRingKeys; k++) { tab.maxs[k] = 0ull; tab.maxdist[k] = 0u; }
  for (int k = 0; k < R; k++) {
    const int base = ring_start[k], m = ring_start[k + 1] - base;
    const float4* ring = bpt.data() + base;
    unsigned maxd_ref = 0u;
    for (int t = 0; t < m; t++) {
      const int idx = URF_F2I(ring[t].w);
      tab.maxs[k] = std::max(tab.maxs[k], planar_sum_bits(ring[t].x, ring[t].y));
      maxd_ref = std::max(maxd_ref, fbits(d2[idx]));
      const bool hit = (prm.x_zero && xzero_mark(prm, ring, m, t, newY.data())) ||
                       (prm.z_zero && (prm.curbPoints == 5 ? zzero_mark_t<5>(prm, ring, m, t) : zzero_mark_t<0>(prm, ring, m, t)));
      if (hit) curb_hit(idx, k);
    }
    tab.maxdist[k] = fbits(maxdist_from_bits(tab.maxs[k]));        // k_tab1
    if (tab.maxdist[k] != maxd_ref) return -102;                   // max of the sums first, one square root after: same value
  }
  if (dbg) {
    for (int i = 0; i < n; i++) {
      if (alpha[i] < 0.0f) continue;
      if (dbg->alpha_v) dbg->alpha_v[i] = alpha[i];
      if (dbg->star_mark) dbg->star_mark[i] = (int8_t)star_mark[i];
      if (ringid[i] < 0) continue;
      if (dbg->az) dbg->az[i] = az[i];
      if (dbg->d2) dbg->d2[i] = d2[i];
      if (dbg->det_label) dbg->det_label[i] = (int8_t)mark[i];
    }
    for (int k = 0; k < R; k++) {
      if (dbg->ring_angle) dbg->ring_angle[k] = tab.angle[k];
      if (dbg->max_dist) dbg->max_dist[k] = bitsf(tab.maxdist[k]);
    }
  }

  // ---- k_tables
  CurbView cv{cmin.data(), cmax.data(), ne.data()};
  for (int k = 0; k < R; k++) {
    unsigned short run = 0;
    for (int bin = 0; bin < kDegBins; bin++) { ne[(size_t)k * (kDegBins + 1) + bin] = run; run += cmin[(size_t)k * kDegBins + bin] != 0x7f800000u; }
    ne[(size_t)k * (kDegBins + 1) + kDegBins] = run;
  }
  std::vector<float> Tf((size_t)kTStride * prm.channels, 0.f), Tb((size_t)kTStride * prm.channels, 0.f);
  SparseMax* spm = new SparseMax();
  {
    const float arc = arc_distance(prm, bitsf(tab.maxdist[0]));
    for (int k = 0; k < R; k++) tab.A[k] = ring_width(arc, bitsf(tab.maxdist[k]));
    for (int w = 0; w < 4; w++) tab.q[w] = blind_quarter(prm, cv, R, w);
    // k_reach: cells (dir, i, k) in parallel on the GPU, minimum kept with atomicMin
    for (int dir = 0; dir < 2; dir++)
      for (int i = 0; i < kDegBins; i++) {
        tab.reach[dir][i] = R;
        if (dir == 0 ? i > prm.fwd_last : i < prm.bwd_first) continue;
        for (int k = R - 1; k >= 0; k--) if (window_blocked(prm, cv, tab.A[k], dir, i, k)) tab.reach[dir][i] = k;
      }
    // k_tab2
    for (int k = 0; k < R; k++) build_T_row(prm, tab.reach[0], tab.reach[1], tab.q, k, tab.A[k], Tf.data() + (size_t)k * kTStride, Tb.data() + (size_t)k * kTStride);
    // cross-check tables: the sequential reach (window_reach) and the window-search formulation of the per-point test
    for (int dir = 0; dir < 2; dir++)
      for (int i = 0; i < kDegBins; i++) {
        const int reach = window_reach(prm, cv, tab.A, tab.q, R, dir, i);
        spm->st[dir][0][i] = (unsigned short)reach;
      }
    for (int l = 1; l < kStLevels; l++)
      for (int dir = 0; dir < 2; dir++)
        for (int i = 0; i < kDegBins; i++) {
          const int j = i + (1 << (l - 1));
          const unsigned short a = spm->st[dir][l - 1][i], c = j < kDegBins ? spm->st[dir][l - 1][j] : (unsigned short)0;
          spm->st[dir][l][i] = a > c ? a : c;
        }
  }

  // ---- k_label (input order), k_dmax, k_best, k_verts
  std::vector<unsigned> dmax(kDegBins, 0u);                     // k_markers1 keeps these two in its shared memory
  std::vector<unsigned long long> best(kDegBins, ~0ull);
  for (int i = 0; i < kDegBins; i++) tab.cutbest[i] = ~0ull;
  int formulation_mismatch = 0;
  std::vector<int> road;
  for (int i = 0; i < n; i++) {
    const int k = ringid[i];
    if (alpha[i] < 0.0f) continue;                       // label stays URF_LABEL_OUTSIDE
    if (k < 0) { if (out->label) out->label[i] = URF_LABEL_NONE; continue; }
    const bool cov = covered_T(Tf.data(), Tb.data(), k, az[i]);
    if (cov != covered_by_window(prm, *spm, tab.A[k], k, az[i])) formulation_mismatch++;
    const int lab = mark[i] == 2 ? 2 : cov ? 1 : 0;
    if (out->label) out->label[i] = lab;
    if (out->ring) out->ring[i] = k;
    if (lab == 1) { out->n_road++; road.push_back(i); } else if (lab == 2) out->n_curb++;
    if (lab != 1 && az[i] >= 0.0f) { const int bin = deg_bin(az[i]); tab.cutbest[bin] = std::min(tab.cutbest[bin], best_key(k, fbits(az[i]), i)); }
  }
  if (formulation_mismatch) return -100;      // threshold tables disagree with the window search: a logic bug
  for (int i : road) {
    if (!(az[i] >= 0.0f)) continue;
    const int bin = deg_bin(az[i]);
    if (marker_candidate(tab.cutbest[bin], ringid[i], fbits(az[i]), i)) dmax[bin] = std::max(dmax[bin], fbits(d2[i]));
  }
  for (int i : road) {
    if (!(az[i] >= 0.0f)) continue;
    const int bin = deg_bin(az[i]);
    if (fbits(d2[i]) != 0u && fbits(d2[i]) == dmax[bin] && marker_candidate(tab.cutbest[bin], ringid[i], fbits(az[i]), i))
      best[bin] = std::min(best[bin], best_key(ringid[i], fbits(az[i]), i));
  }
  int cM = 0;
  for (int i = 0; i < kDegBins; i++) {
    if (best[i] == ~0ull) continue;
    const int p = (int)(best[i] & 0xffffffull);
    out->vert[cM][0] = xyzi[4 * p]; out->vert[cM][1] = xyzi[4 * p + 1]; out->vert[cM][2] = xyzi[4 * p + 2];
    out->vert[cM][3] = tab.cutbest[i] != ~0ull ? 1.0f : 0.0f;
    cM++;
  }
  out->n_vert = cM;
  delete spm;

  // ---- k_sort_rings
  for (int k = 0; k < R; k++) {
    const int base = ring_start[k], m = ring_start[k + 1] - base;
    std::vector<unsigned long long> keys(m);
    for (int t = 0; t < m; t++) keys[t] = ((unsigned long long)fbits(az[URF_F2I(bpt[base + t].w)]) << 32) | (unsigned)t;
    std::sort(keys.begin(), keys.end());
    for (int t = 0; t < m; t++) {
      if (out->order) out->order[base + t] = URF_F2I(bpt[base + (unsigned)keys[t]].w);
      if (t > 0 && (unsigned)(keys[t - 1] >> 32) == (unsigned)(keys[t] >> 32)) flags |= F_TIE_AZIMUTH;
    }
  }
  out->n_rings = R; out->n_order = N;
  if (out->ring_start) for (int k = 0; k <= kRingKeys; k++) out->ring_start[k] = ring_start[k];
  out->flags = flags;   // the model reports internal bits too (tests look at F_SPEC_VIOLATION / F_EXACT_REG)
  delete tabp;
  return 0;
}
