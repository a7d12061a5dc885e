// tests/kat/star_prefix_check.cpp — host check of the near-first star sort's exactness argument (k_star_sort_warp /
// k_star_scan / k_star_refine in urf_kernels.cuh), with the same arithmetic functions the kernels call
// (urf_logic.cuh): for random sectors, "sort everything, walk until the first edge" (star_shaped_search.cpp:109-150) must
// mark the same point as "split at the sampled pivot, sort and walk the near part, and if no edge was found sort the
// points ABOVE the prefix's largest radius behind the prefix (that must be exactly the rest, and give the full order) and
// resume the walk there from the saved running mean / deviation, slopes and reciprocals computed per point up front"
// (k_star_refine's select_far + star_resume_walk_warp).
// usage: star_prefix_check <sectors> <seed>   -> prints "sectors=.. hits=.. prefix_hits=.. refined=.. mismatches=.."
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <vector>
#include <cuda_runtime.h>   // float4 only
#include "../../urban_road_filter_b200/csrc/urf_logic.cuh"
#include "../../urban_road_filter_b200/csrc/urf_host.hpp"

using namespace urf;

int main(int argc, char** argv) {
  const int sectors = argc > 1 ? atoi(argv[1]) : 20000;
  std::mt19937 g(argc > 2 ? atoi(argv[2]) : 1);
  urf_params up;
  memset(&up, 0, sizeof(up));                               // only the star-search parameters matter here
  up.star_shaped_method = 1; up.beamZone = 30; up.curb_points = 5; up.channels = 64; up.interval = 0.18;
  long hits = 0, prefix_hits = 0, refined = 0, bad = 0;
  for (int t = 0; t < sectors; t++) {
    // parameter and geometry variety: flat ground with noise, optional curb step at a random radius, optional wall
    up.curb_slope_deg = std::uniform_real_distribution<double>(5, 80)(g);
    up.kdev_param = std::uniform_real_distribution<double>(0.2, 3)(g);
    up.kdist_param = std::uniform_real_distribution<double>(0.5, 8)(g);
    up.dmin_param = std::uniform_int_distribution<int>(1, 40)(g);
    DevParams prm{};
    narrow_params(&up, &prm, 57.2957802f, 0, 0);
    const int n = std::uniform_int_distribution<int>(129, 1024)(g);
    const float rmax = std::uniform_real_distribution<float>(5.f, 80.f)(g);
    const float curb_r = std::uniform_real_distribution<float>(0.f, 1.4f)(g) * rmax;     // beyond rmax: no curb at all
    const float noise = std::uniform_real_distribution<float>(0.f, 0.02f)(g);
    std::vector<float4> pts(n);
    std::uniform_real_distribution<float> U(0.3f, rmax), N(-1.f, 1.f);
    for (int i = 0; i < n; i++) {
      const float r = U(g);
      float z = -1.8f + noise * N(g);
      if (r > curb_r) z += 0.12f;
      if (r > 0.9f * rmax && (t & 3) == 0) z += (r - 0.9f * rmax) * 3.f;               // a wall face
      pts[i] = make_float4(r, z, bitsf((unsigned)i), 0.f);
    }
    auto by_r = [](const float4& a, const float4& b) { return a.x < b.x || (a.x == b.x && fbits(a.z) < fbits(b.z)); };   // (r, input index)
    // (1) the reference's way
    std::vector<float4> full = pts;
    std::sort(full.begin(), full.end(), by_r);
    const int hit_full = star_scan_sector(prm, full.data(), n);
    // (2) near-first, as the kernels do it
    unsigned samples[32];
    for (int l = 0; l < 32; l++) samples[l] = fbits(pts[(int)(((unsigned)l * (unsigned)n) >> 5)].x);
    unsigned pivot = 0;
    for (int l = 0; l < 32; l++) {
      int rank = 0;
      for (int j = 0; j < 32; j++) rank += (samples[j] < samples[l]) || (samples[j] == samples[l] && j < l);
      if (rank == kStarPivot) pivot = samples[l];
    }
    std::vector<float4> near;
    for (const float4& p : pts) if (fbits(p.x) < pivot) near.push_back(p);
    const int m = (int)near.size();
    long mark_nf = -1;                                        // input index of the point near-first marks
    if (m >= 32 && 4 * m <= 3 * n) {
      std::sort(near.begin(), near.end(), by_r);
      StarState st;
      star_init(st, near[0].x, near[0].y);
      int hit = -1;
      for (int i = 1; i < m && hit < 0; i++) if (star_step(prm, st, i, near[i].x, near[i].y)) hit = i;
      if (hit >= 0) { prefix_hits++; mark_nf = fbits(near[hit].z); }
      else {                                                  // resume on the full order from the saved state
        refined++;
        const unsigned kmax = fbits(near[m - 1].x);           // select_far: everything above the prefix's largest radius
        std::vector<float4> far;
        for (const float4& p : pts) if (fbits(p.x) > kmax) far.push_back(p);
        std::sort(far.begin(), far.end(), by_r);
        std::vector<float4> all = near;
        all.insert(all.end(), far.begin(), far.end());
        bool same = (int)all.size() == n;
        for (int i = 0; same && i < n; i++) same = fbits(all[i].x) == fbits(full[i].x) && fbits(all[i].z) == fbits(full[i].z);
        if (!same) { if (bad < 5) fprintf(stderr, "sector %d: prefix + sorted rest is not the full order (n=%d m=%d rest=%zu)\n", t, n, m, far.size()); bad++; continue; }
        StarState rs;
        rs.avg = st.avg; rs.dev = st.dev; rs.nan = st.nan; rs.bx = 0.f; rs.by = 0.f;
        for (int i = m; i < n && hit < 0; i++) {              // star_resume_walk_warp: per-point part first, then the recurrence
          float dx;
          const float slp = star_slope(all[i - 1].x, all[i - 1].y, all[i].x, all[i].y, &dx);
          if (star_update(prm, rs, i, slp, URF_FMUL(dx, prm.kdist), star_inv(i))) hit = i;
        }
        if (hit >= 0) mark_nf = fbits(all[hit].z);
      }
    } else {
      if (hit_full >= 0) mark_nf = fbits(full[hit_full].z);   // the kernel sorts the whole sector in this case
    }
    if (hit_full >= 0) hits++;
    const long mark_full = hit_full >= 0 ? (long)fbits(full[hit_full].z) : -1;
    if (mark_full != mark_nf) { if (bad < 5) fprintf(stderr, "sector %d: n=%d m=%d full marks %ld, near-first marks %ld\n", t, n, m, mark_full, mark_nf); bad++; }
  }
  printf("sectors=%d hits=%ld prefix_hits=%ld refined=%ld mismatches=%ld\n", sectors, hits, prefix_hits, refined, bad);
  return bad != 0;
}
