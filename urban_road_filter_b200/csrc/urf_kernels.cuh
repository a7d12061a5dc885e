// urf_kernels.cuh — sm_100a kernels of the per-scan road/curb classification path (pipeline v2).
//
// Every kernel takes the batch index from blockIdx.y (or blockIdx.x for one-CTA-per-scan kernels): a launch covers a
// whole batch of scans laid out back to back with `S` points of stride. Everything that decides a label is computed by
// the host+device functions of urf_logic.cuh (bit-identical to the x86-64 -O2 build of the reference, file:line cited
// there); the kernels add indexing, staging, atomics and synchronisation.
//
// Pipeline (DESIGN.md has the picture):
//   k_reset -> k_points -> k_register -> k_assign -> k_scan_offsets (+ exact re-registration of refuted scans)
//   -> k_scatter -> k_star_sort_warp (near-first) -> k_star_sort_big (large sectors, exact fallback) -> k_star_scan
//   -> k_star_refine (sectors without an edge in their prefix: full sort, walk resumed)
//   -> k_ring_detect4 / k_ring_detect (on a side stream, next to the star-shaped search) -> k_tab1 -> k_reach -> k_tab2
//   -> k_label (input order) -> k_markers1 (one CTA per scan; scans above 300 k points: k_markers_grid x 2 -> k_verts)
//   [-> k_sort_rings when the emission order is requested]
//   PointCloud2 entry points: k_unpack_cloud2 in front, k_pack_count -> k_pack_scan -> k_pack_write behind
#pragma once
#include <type_traits>

#include "urf_device.cuh"
#include "urf_logic.cuh"
#include "urf_stdsort.cuh"

namespace urf {

__constant__ float c_beam_d[kSectKeys];
__constant__ float c_beam_o[kSectKeys];
__constant__ unsigned char c_beam_yx[kSectKeys];

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
// 32-bit offset of scan b inside the batch-major arrays (urf_create keeps max_batch * max_points below 2^31): array
// accesses then cost one IMAD.WIDE instead of 64-bit multiply/add chains
__device__ __forceinline__ unsigned scan_base(int b, int S) { return (unsigned)b * (unsigned)S; }

// CTA-wide bitonic sort of npad (power of two) keys in shared or global memory; all threads must call.
template <class T>
__device__ void cta_bitonic(T* a, int npad) {
  for (int k = 2; k <= npad; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < (npad >> 1); t += blockDim.x) {
        int i = 2 * t - (t & (j - 1));
        int l = i + j;
        bool up = (i & k) == 0;
        T x = a[i], y = a[l];
        if ((x > y) == up) { a[i] = y; a[l] = x; }
      }
      __syncthreads();
    }
  }
}

__device__ __forceinline__ int next_pow2(int n) { int p = 1; while (p < n) p <<= 1; return p; }

// A detector found input point idx of scan b to be a curb point (star_shaped_search.cpp:146, x_zero_method.cpp:66,
// z_zero_method.cpp:71): mark it and, if it sits in a ring bucket (k = its ring, or -1 = look it up), enter its azimuth
// into the curb aggregates of that ring's integer-degree bin — what blindSpots reads. NaN azimuths fall out.
__device__ __forceinline__ void curb_hit(const DevBuffers& buf, const DevParams& prm, int b, unsigned gb, int idx, int k) {
  buf.mark[gb + (unsigned)idx] = 2;
  if (k < 0) k = buf.ringid[gb + (unsigned)idx];
  if (k < 0) return;                                   // not in array3D: the mark is never read (lidar_segmentation.cpp:241)
  const float a = buf.az[gb + (unsigned)idx];
  if (a >= 0.0f) {
    const unsigned o = ((unsigned)b * (unsigned)prm.channels + (unsigned)k) * kDegBins + (unsigned)deg_bin(a);
    atomicMin(&buf.cmin[o], fbits(a));
    atomicMax(&buf.cmax[o], fbits(a));
  }
}
// ring of bucket position p: rings are contiguous in bucket order, ring_start has kRingKeys + 1 non-decreasing entries
__device__ __forceinline__ int ring_of_position(const int* __restrict__ ring_start, int p) {
  int lo = 0, hi = kRingKeys;
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (ring_start[mid] <= p) lo = mid + 1; else hi = mid; }
  return lo - 1;
}

// ---------------------------------------------------------------------------------------------------------------------
// k_reset: per-call initialisation of the per-scan tables.
__global__ void k_reset(DevBuffers buf, DevParams prm) {
  const int b = blockIdx.y;
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const int nth = gridDim.x * blockDim.x;
  ScanOut& o = buf.out[b];
  ScanTab& t = buf.tab[b];
  if (tid == 0) {
    o.n_in = buf.n[b]; o.n_roi = 0; o.n_rings = 0; o.n_order = 0; o.n_road = 0; o.n_curb = 0; o.n_vert = 0; o.flags = 0;
  }
  for (int i = tid; i <= kRingKeys; i += nth) o.ring_start[i] = 0;
  for (int i = tid; i < kRingKeys; i += nth) { t.maxs[i] = 0ull; t.maxdist[i] = 0u; t.angle[i] = 0.f; t.regidx[i] = 0x7fffffff; t.regorder[i] = 0x7fffffff; }
  for (int i = tid; i < kDegBins; i += nth) { t.cutbest[i] = ~0ull; t.dmax[i] = 0u; t.best[i] = ~0ull; }
  for (int i = tid; i < kSectKeys; i += nth) t.sect_cnt[i] = 0;
  if (tid == 0) { t.nbig = 0; t.nslow = 0; t.nrefine = 0; }
  unsigned* fi = buf.firstidx + (size_t)b * (kElevBins + 1);
  for (int i = tid; i <= kElevBins; i += nth) fi[i] = 0xffffffffu;
  const size_t nb = (size_t)prm.channels * kDegBins;
  unsigned* cmin = buf.cmin + (size_t)b * nb;
  unsigned* cmax = buf.cmax + (size_t)b * nb;
  for (size_t i = tid; i < nb; i += nth) { cmin[i] = 0x7f800000u; cmax[i] = 0u; }
}

// ---------------------------------------------------------------------------------------------------------------------
// k_points: everything that depends on one input point alone — ROI crop predicate, range and elevation angle
// (lidar_segmentation.cpp:106-113,148-166), planar range and azimuth (:245-269; the squares are shared with the range) and
// the star sector (star_shaped_search.cpp:164-173). Also records, per fine elevation bin, the first input index that
// falls into it (speculation input for k_register).
__global__ void __launch_bounds__(256) k_points(DevBuffers buf, DevParams prm, int S) {
  const int b = blockIdx.y;
  const int n = buf.n[b];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  int keep = 0, sec = -1;
  if (i < n) {
    const unsigned g = scan_base(b, S) + (unsigned)i;
    const float4 p = __ldg(&buf.in[g]);
    keep = roi_keep(prm, p.x, p.y, p.z);
    float a = -1.0f;
    if (keep) {
      float d, az;
      point_angles(p.x, p.y, p.z, &a, &d, &az);
      unsigned* fi = buf.firstidx + (size_t)b * (kElevBins + 1) + elev_bin(a);
      if (*fi > (unsigned)i) atomicMin(fi, (unsigned)i);      // plain (possibly stale) read: a stale value is only larger
      if (a == 0.0f) atomicOr(&buf.out[b].flags, F_ZERO_ALPHA);
      if (az != az) atomicOr(&buf.out[b].flags, F_NAN_AZIMUTH);   // x == y == 0 inside the ROI
      if (prm.star) sec = star_sector(prm, p.x, p.y, c_beam_d, c_beam_o, c_beam_yx);   // star_shaped_search.cpp:164-173
      buf.az[g] = az;
      buf.d2[g] = d;
    }
    buf.alpha_v[g] = a;
    buf.mark[g] = 0;
    buf.sect[g] = (short)sec;
  }
  const unsigned bal = __ballot_sync(0xffffffffu, keep);
  if (lane_id() == 0 && bal) atomicAdd(&buf.out[b].n_roi, __popc(bal));
  // per-sector point counts of the (unordered) sector partition: one atomic per group of equal sectors in the warp
  const unsigned peers = __match_any_sync(0xffffffffu, sec);
  if (sec >= 0 && lane_id() == __ffs(peers) - 1) atomicAdd(&buf.tab[b].sect_cnt[sec], __popc(peers));
}

// ---------------------------------------------------------------------------------------------------------------------
// Ring registration, lidar_segmentation.cpp:136-139,170-196: a point registers its elevation angle iff no VISIBLE
// registered angle lies within `interval` of it and fewer than `channels` angles are registered. "Visible": the
// reference's scan stops at the first angle[j] == 0, so once an angle of exactly 0 is registered, it and everything
// registered after it are never compared again.
//
// Exact path (any input): rounds of "find the first uncovered point after the last registrant" with a CTA-wide min.
__device__ void register_exact_cta(const float* __restrict__ alpha, int n, float interval, int channels, float* s_vis,
                                   float* s_reg, int* s_idx, int* s_red, int* out_m) {
  __shared__ int s_min;
  int m = 0, vis = 0, i_last = -1;
  bool frozen = false;
  while (m < channels) {
    int local = 0x7fffffff;
    for (int i = i_last + 1 + threadIdx.x; i < n; i += blockDim.x) {
      const float a = alpha[i];
      if (a < 0.0f) continue;
      bool cov = false;
      for (int t = 0; t < vis; t++) {
        if (fabsf(__fsub_rn(s_vis[t], a)) <= interval) { cov = true; break; }   // :179
      }
      if (!cov) { local = i; break; }
    }
    for (int o = 16; o > 0; o >>= 1) local = min(local, __shfl_xor_sync(0xffffffffu, local, o));
    if (lane_id() == 0) s_red[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0) {
      int v = 0x7fffffff;
      for (int w = 0; w < (int)(blockDim.x >> 5); w++) v = min(v, s_red[w]);
      s_min = v;
    }
    __syncthreads();
    const int istar = s_min;
    __syncthreads();
    if (istar == 0x7fffffff) break;
    const float a = alpha[istar];
    if (threadIdx.x == 0) { s_reg[m] = a; s_idx[m] = istar; if (!frozen && a != 0.0f) s_vis[vis] = a; }
    if (!frozen) { if (a == 0.0f) frozen = true; else vis++; }
    m++;
    i_last = istar;
    __syncthreads();
  }
  *out_m = m;
}

// Sort the m registered (angle, regidx) pairs by angle (:205), publish them and build the elevation-bin lookup table
// k_assign starts its ring search from. Angles are >= 0 so their bits order them.
__device__ void publish_rings_cta(ScanTab& tab, ScanOut& out, unsigned short* lut, float interval, const float* s_reg,
                                  const int* s_idx, int m, unsigned long long* s_keys, float* s_sorted) {
  for (int t = threadIdx.x; t < kRingKeys; t += blockDim.x)
    s_keys[t] = t < m ? (((unsigned long long)fbits(s_reg[t]) << 32) | (unsigned)s_idx[t]) : ~0ull;
  __syncthreads();
  cta_bitonic(s_keys, kRingKeys);
  for (int t = threadIdx.x; t < kRingKeys; t += blockDim.x) {
    if (t < m) {
      const float a = bitsf((unsigned)(s_keys[t] >> 32));
      s_sorted[t] = a;
      tab.angle[t] = a;
      tab.regidx[t] = (int)(unsigned)s_keys[t];
      tab.regorder[t] = s_idx[t];
    } else { s_sorted[t] = 0.f; tab.angle[t] = 0.f; tab.regidx[t] = 0x7fffffff; tab.regorder[t] = 0x7fffffff; }
  }
  if (threadIdx.x == 0) out.n_rings = m;
  __syncthreads();
  for (int e = threadIdx.x; e <= kElevBins; e += blockDim.x) lut[e] = (unsigned short)ring_lut_entry(s_sorted, m, interval, e);
}

// k_register: one CTA (256 threads) per scan. Fast path: the greedy registration is run over "candidates" only — the
// first point of every non-empty fine elevation bin, in input order. That is a speculation (a registrant need not be
// the first of its bin); k_assign verifies it against every point and k_scan_offsets repairs a failed speculation (exact greedy, in-kernel).
__global__ void __launch_bounds__(256) k_register(DevBuffers buf, DevParams prm, int S) {
  const int b = blockIdx.x;
  const int n = buf.n[b];
  ScanOut& out = buf.out[b];
  ScanTab& tab = buf.tab[b];
  const float* alpha = buf.alpha_v + (size_t)b * S;
  __shared__ unsigned s_cand[kMaxCand];
  __shared__ float s_calpha[kMaxCand];
  __shared__ float s_vis[kRingKeys];
  __shared__ float s_reg[kRingKeys];
  __shared__ float s_sorted[kRingKeys];
  __shared__ int s_idx[kRingKeys];
  __shared__ unsigned long long s_keys[kRingKeys];
  __shared__ int s_red[8];
  __shared__ int s_cnt, s_m;
  if (out.n_roi < 30) {                      // lidar_segmentation.cpp:124-126: nothing happens for this scan
    if (threadIdx.x == 0) out.n_rings = 0;
    return;
  }
  bool exact = prm.force_exact || (out.flags & F_ZERO_ALPHA);
  if (!exact) {
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    const unsigned* fi = buf.firstidx + (size_t)b * (kElevBins + 1);
    for (int t = threadIdx.x; t <= kElevBins; t += blockDim.x) {
      const unsigned v = fi[t];
      if (v != 0xffffffffu) { int s = atomicAdd(&s_cnt, 1); if (s < kMaxCand) s_cand[s] = v; }
    }
    __syncthreads();
    const int cnt = s_cnt;
    if (cnt > kMaxCand) exact = true;        // uniform across the CTA
    else {
      const int npad = next_pow2(cnt < 2 ? 2 : cnt);
      for (int t = cnt + threadIdx.x; t < npad; t += blockDim.x) s_cand[t] = 0xffffffffu;
      __syncthreads();
      cta_bitonic(s_cand, npad);
      for (int t = threadIdx.x; t < cnt; t += blockDim.x) s_calpha[t] = alpha[s_cand[t]];
      __syncthreads();
      if (threadIdx.x < 32) {
        int m = 0;
        for (int c = 0; c < cnt && m < prm.channels; c++) {
          const float a = s_calpha[c];
          bool cov = false;
          for (int t = lane_id(); t < m; t += 32)
            if (fabsf(__fsub_rn(s_reg[t], a)) <= prm.interval) cov = true;          // :179
          cov = __any_sync(0xffffffffu, cov);
          if (!cov) {
            if (lane_id() == 0) { s_reg[m] = a; s_idx[m] = (int)s_cand[c]; }
            m++;
            __syncwarp();
          }
        }
        if (lane_id() == 0) s_m = m;
      }
      __syncthreads();
    }
  }
  if (exact) {
    int m;
    register_exact_cta(alpha, n, prm.interval, prm.channels, s_vis, s_reg, s_idx, s_red, &m);
    if (threadIdx.x == 0) { s_m = m; atomicOr(&out.flags, F_EXACT_REG); }
    __syncthreads();
  }
  publish_rings_cta(tab, out, buf.lut + (size_t)b * (kElevBins + 1), prm.interval, s_reg, s_idx, s_m, s_keys, s_sorted);
}

// ---------------------------------------------------------------------------------------------------------------------
// k_assign: per input point — ring index (lidar_segmentation.cpp:226-233: first sorted angle within `interval`) and the
// per-warp-chunk ring histogram of the stable ring partition. assign_chunk is one warp's chunk of kChunk points; cnt is
// the warp's zeroed shared histogram. Returns true (per lane) where the speculated registration is refuted.
__device__ __forceinline__ bool assign_chunk(const DevBuffers& buf, const DevParams& prm, int b, int S, int T, int chunk, int n, bool live,
                                             bool verify, const float* s_angle, const int* s_regidx, const int* regorder, int R,
                                             const unsigned short* __restrict__ lut, unsigned* cnt, int lane) {
  bool violation = false;
  // two halves of eight iterations: the eight elevation loads are issued together, then the eight table look-ups they
  // address, and only then the (short, shared-memory) ring searches — two memory round trips per half instead of sixteen
  constexpr int H = 8;
  static_assert((kChunk / 32) % H == 0, "chunk iterations come in groups of H");
#pragma unroll 1
  for (int h0 = 0; h0 < kChunk / 32; h0 += H) {
    float av[H];
    unsigned short start[H];
#pragma unroll
    for (int u = 0; u < H; u++) {
      const int i = chunk * kChunk + (h0 + u) * 32 + lane;
      av[u] = i < n ? buf.alpha_v[scan_base(b, S) + (unsigned)i] : -1.0f;
    }
#pragma unroll
    for (int u = 0; u < H; u++) start[u] = (live && av[u] >= 0.0f) ? lut[elev_bin(av[u])] : (unsigned short)0;
#pragma unroll
    for (int u = 0; u < H; u++) {
      const int i = chunk * kChunk + (h0 + u) * 32 + lane;
      int ring = -1;
      if (i < n) {
        const float a = av[u];
        const bool kept = live && a >= 0.0f;
        if (kept) {
          int lo;
          ring = assign_ring_from(s_angle, R, a, prm.interval, start[u], &lo);
          if (verify && registration_violation(s_angle, s_regidx, regorder, R, prm.channels, prm.interval, a, i, lo)) violation = true;
        }
        buf.ringid[scan_base(b, S) + (unsigned)i] = kept ? (short)ring : (short)-2;   // -2: not part of the ROI cloud (k_label writes URF_LABEL_OUTSIDE)
      }
      // histogram: a ring-major scan puts one ring into a warp (one add of 32), a column-major one 32 different rings
      // (32 conflict-free shared atomics); results unused, so no read-modify-write chain between iterations
      const int ring0 = __shfl_sync(0xffffffffu, ring, 0);
      if (__all_sync(0xffffffffu, ring == ring0)) { if (lane == 0 && ring0 >= 0) atomicAdd(&cnt[ring0], 32u); }
      else if (ring >= 0) atomicAdd(&cnt[ring], 1u);
    }
  }
  __syncwarp();
  unsigned* row = buf.hist + ((size_t)b * T + chunk) * kRingKeys;
  for (int t = lane; t < kRingKeys; t += 32) row[t] = cnt[t];
  return violation;
}

__global__ void __launch_bounds__(kWarpsPerBlock * 32) k_assign(DevBuffers buf, DevParams prm, int S, int T) {
  const int b = blockIdx.y;
  ScanOut& out = buf.out[b];
  const int flags = out.flags;
  const int n = buf.n[b];
  const int warp = threadIdx.x >> 5, lane = lane_id();
  const int chunk = blockIdx.x * kWarpsPerBlock + warp;
  __shared__ float s_angle[kRingKeys];
  __shared__ int s_regidx[kRingKeys];
  __shared__ unsigned s_cnt[kWarpsPerBlock][kRingKeys];
  ScanTab& tab = buf.tab[b];
  const int R = out.n_rings;
  for (int t = threadIdx.x; t < kRingKeys; t += blockDim.x) { s_angle[t] = tab.angle[t]; s_regidx[t] = tab.regidx[t]; }
  for (int t = lane; t < kRingKeys; t += 32) s_cnt[warp][t] = 0;
  __syncthreads();
  if (chunk * kChunk >= n) return;             // whole warp; no block-level sync follows
  const bool violation = assign_chunk(buf, prm, b, S, T, chunk, n, out.n_roi >= 30, !(flags & F_EXACT_REG), s_angle, s_regidx, tab.regorder, R,
                                      buf.lut + (size_t)b * (kElevBins + 1), s_cnt[warp], lane);
  if (__any_sync(0xffffffffu, violation) && lane == 0) atomicOr(&out.flags, F_SPEC_VIOLATION);
}

// ---------------------------------------------------------------------------------------------------------------------
// k_scan_offsets: one CTA (1024 threads) per scan turns hist[chunk][ring] into exclusive scatter offsets (ring-major
// bases + prefix over chunks), publishes ring_start, and turns the sector counts into sect_start + scatter cursors.
// In front of that it repairs a scan whose speculated registration k_assign refuted (F_SPEC_VIOLATION, rare): the exact
// registration, then ring ids and chunk histograms of the whole scan again, one chunk per warp at a time.
__global__ void __launch_bounds__(1024) k_scan_offsets(DevBuffers buf, DevParams prm, int S, int T) {
  __shared__ unsigned s_part[32][kRingKeys];     // per-warp partial sums, then per-warp exclusive prefixes
  __shared__ unsigned s_base[kRingKeys];
  const int b = blockIdx.x;
  const int n = buf.n[b];
  const int rows = (n + kChunk - 1) / kChunk;
  const int warp = threadIdx.x >> 5, lane = lane_id();
  {
    ScanOut& out = buf.out[b];
    const int flags = out.flags;
    if ((flags & F_SPEC_VIOLATION) && !(flags & F_EXACT_REG)) {      // uniform across the CTA
      __shared__ float s_vis[kRingKeys], s_reg[kRingKeys], s_sorted[kRingKeys];
      __shared__ int s_idx[kRingKeys];
      __shared__ unsigned long long s_keys[kRingKeys];
      __shared__ int s_red[32];
      __shared__ int s_m;
      int m;
      register_exact_cta(buf.alpha_v + (size_t)b * S, n, prm.interval, prm.channels, s_vis, s_reg, s_idx, s_red, &m);
      if (threadIdx.x == 0) s_m = m;
      __syncthreads();
      const unsigned short* lut = buf.lut + (size_t)b * (kElevBins + 1);
      publish_rings_cta(buf.tab[b], out, buf.lut + (size_t)b * (kElevBins + 1), prm.interval, s_reg, s_idx, s_m, s_keys, s_sorted);
      __syncthreads();                                                // s_sorted = the sorted angles, lut written
      const int R = s_m;
      for (int c0 = 0; c0 < rows; c0 += 32) {
        for (int t = lane; t < kRingKeys; t += 32) s_part[warp][t] = 0;
        __syncwarp();
        if (c0 + warp < rows) assign_chunk(buf, prm, b, S, T, c0 + warp, n, true, false, s_sorted, nullptr, nullptr, R, lut, s_part[warp], lane);
        __syncwarp();
      }
      if (threadIdx.x == 0) out.flags = flags | F_EXACT_REG;
      __syncthreads();                                                // the histogram rows are read back below
    }
  }
  const int rpw = (rows + 31) / 32;
  const int r0 = min(rows, warp * rpw), r1 = min(rows, (warp + 1) * rpw);
  unsigned* hist = buf.hist + (size_t)b * T * kRingKeys;
  for (int key = lane; key < kRingKeys; key += 32) {
    unsigned s = 0;
    for (int r = r0; r < r1; r++) s += hist[(size_t)r * kRingKeys + key];
    s_part[warp][key] = s;
  }
  __syncthreads();
  if (threadIdx.x < kRingKeys) {
    unsigned run = 0;
    for (int w = 0; w < 32; w++) { unsigned v = s_part[w][threadIdx.x]; s_part[w][threadIdx.x] = run; run += v; }
    s_base[threadIdx.x] = run;                  // total of this ring
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned run = 0;
    ScanOut& o = buf.out[b];
    for (int k = 0; k < kRingKeys; k++) { unsigned v = s_base[k]; s_base[k] = run; o.ring_start[k] = (int)run; run += v; }
    o.ring_start[kRingKeys] = (int)run;
    o.n_order = (int)run;
  } else if (threadIdx.x == 32) {
    ScanTab& t = buf.tab[b];
    int run = 0;
    for (int k = 0; k < kSectKeys; k++) { const int v = t.sect_cnt[k]; t.sect_start[k] = run; t.sect_cur[k] = run; run += v; }
    t.sect_start[kSectKeys] = run;
  }
  __syncthreads();
  for (int key = lane; key < kRingKeys; key += 32) {
    unsigned run = s_base[key] + s_part[warp][key];
    for (int r = r0; r < r1; r++) {
      unsigned* p = &hist[(size_t)r * kRingKeys + key];
      unsigned v = *p; *p = run; run += v;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// k_scatter: stable scatter of every point into its ring bucket (input order inside a ring, lidar_segmentation.cpp:221-
// 277) and unordered scatter into its star sector (the radius sort that follows breaks ties by input index, which is the
// push_back order of star_shaped_search.cpp:173). One warp per chunk of kChunk points, kWarpsPerBlock chunks per CTA.
// Sectors: every point takes a rank inside its sector from a CTA-wide shared counter; after a barrier one thread per
// sector that occurs in the CTA reserves the CTA's slots from the scan's sector cursor with ONE global atomic (all of them
// in flight together), and after a second barrier the records are written to base + rank.
// Ring buckets are written coalesced: the warp first ranks its chunk by ring in shared memory, then walks the chunk in
// ring order so that consecutive lanes write consecutive bucket slots.
__global__ void __launch_bounds__(kWarpsPerBlock * 32) k_scatter(DevBuffers buf, DevParams prm, int S, int T) {
  const int b = blockIdx.y;
  const int n = buf.n[b];
  const int warp = threadIdx.x >> 5, lane = lane_id();
  const int chunk = blockIdx.x * kWarpsPerBlock + warp;
  __shared__ unsigned s_delta[kWarpsPerBlock][kChunk];            // bucket slot of ring-ordered slot t, minus t
  __shared__ unsigned s_lcnt[kWarpsPerBlock][kRingKeys];          // per-ring count, then exclusive local start
  __shared__ unsigned short s_perm[kWarpsPerBlock][kChunk];       // chunk-local point index in ring order
  __shared__ int s_scnt[kSectKeys], s_sbase[kSectKeys];           // sector: points of this CTA, first slot reserved for them
  unsigned* delta = s_delta[warp];
  unsigned* lcnt = s_lcnt[warp];
  unsigned short* perm = s_perm[warp];
  ScanTab& tab = buf.tab[b];
  const bool live = chunk * kChunk < n;                           // a warp past the end only takes part in the barriers
  const unsigned* row = buf.hist + ((size_t)b * T + chunk) * kRingKeys;
  for (int t = threadIdx.x; t < kSectKeys; t += blockDim.x) s_scnt[t] = 0;
  for (int t = lane; t < kRingKeys; t += 32) lcnt[t] = 0;
  __syncthreads();
  const unsigned lt = (1u << lane) - 1u;
  unsigned packed[kChunk / 32];                 // (ring + 1) << 16 | rank inside the chunk's ring group
  unsigned spack[kChunk / 32];                  // (sector + 1) << 16 | rank inside the CTA's sector group
  const unsigned gb = scan_base(b, S), g0 = gb + (unsigned)chunk * kChunk;
  if (live) {
    // groups of 4 iterations: the ring / sector loads of a group are issued together before anything depends on them
    constexpr int GRP = 4;
#pragma unroll
    for (int h = 0; h < kChunk / 32 / GRP; h++) {
      short rr[GRP], ss[GRP];
#pragma unroll
      for (int u = 0; u < GRP; u++) {
        const int li = (h * GRP + u) * 32 + lane;
        const bool in = chunk * kChunk + li < n;
        rr[u] = in ? buf.ringid[g0 + li] : (short)-1;
        ss[u] = in ? buf.sect[g0 + li] : (short)-1;
      }
#pragma unroll
      for (int u = 0; u < GRP; u++) {
        const int it = h * GRP + u;
        // sector rank (any order will do): one shared atomic for a warp that sits in one sector (column-major scans: 32
        // rings of one azimuth), else one per lane
        const int sec = ss[u];
        const int sec0 = __shfl_sync(0xffffffffu, sec, 0);
        int srank = 0;
        if (__all_sync(0xffffffffu, sec == sec0)) {
          int sb = 0;
          if (lane == 0 && sec0 >= 0) sb = atomicAdd(&s_scnt[sec0], 32);
          srank = __shfl_sync(0xffffffffu, sb, 0) + lane;
        } else if (sec >= 0) srank = atomicAdd(&s_scnt[sec], 1);
        spack[it] = sec >= 0 ? (((unsigned)(sec + 1) << 16) | (unsigned)srank) : 0u;
        // stable rank inside the ring: the group's first lane takes the group's slots from the warp's ring counter with a
        // shared atomic (same-address atomics of one warp apply in program order, so iteration order = input order; nothing
        // else orders the iterations, the sixteen of them pipeline), lanes add their position inside the group
        // groups of equal rings in the warp. The two sensor layouts need no MATCH (its latency was the kernel's largest
        // stall): ring-major input puts ONE ring into a warp, column-major input 32 DIFFERENT rings in ascending or
        // descending order (all distinct: every lane is its own group); anything else takes __match_any_sync
        const int ring = rr[u];
        const int rprev = __shfl_up_sync(0xffffffffu, ring, 1), ring0 = __shfl_sync(0xffffffffu, ring, 0);
        unsigned peers;
        if (__all_sync(0xffffffffu, ring == ring0)) peers = 0xffffffffu;
        else if (__all_sync(0xffffffffu, lane == 0 || ring > rprev) || __all_sync(0xffffffffu, lane == 0 || ring < rprev)) peers = 1u << lane;
        else peers = __match_any_sync(0xffffffffu, ring);
        const int leader = __ffs(peers) - 1;
        unsigned rb = 0;
        if (ring >= 0 && lane == leader) rb = atomicAdd(&lcnt[ring], (unsigned)__popc(peers));
        rb = __shfl_sync(0xffffffffu, rb, leader);
        packed[it] = ring >= 0 ? (((unsigned)(ring + 1) << 16) | (rb + __popc(peers & lt))) : 0u;
      }
    }
  }
  __syncthreads();
  for (int t = threadIdx.x; t < kSectKeys; t += blockDim.x) {     // one reservation per sector present in this CTA
    const int c = s_scnt[t];
    s_sbase[t] = c > 0 ? atomicAdd(&tab.sect_cur[t], c) : 0;
  }
  int total = 0;
  if (live) {
    // exclusive scan of the chunk's ring counts -> local starts (runs while the reservations are in flight)
    {
      unsigned v[kRingKeys / 32], sum = 0;
#pragma unroll
      for (int j = 0; j < kRingKeys / 32; j++) { v[j] = lcnt[lane * (kRingKeys / 32) + j]; sum += v[j]; }
      unsigned inc = sum;
      for (int o = 1; o < 32; o <<= 1) { unsigned t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
      unsigned run = inc - sum;
      __syncwarp();
#pragma unroll
      for (int j = 0; j < kRingKeys / 32; j++) { lcnt[lane * (kRingKeys / 32) + j] = run; run += v[j]; }
    }
    __syncwarp();
#pragma unroll
    for (int it = 0; it < kChunk / 32; it++) {
      const unsigned pk = packed[it];
      if (pk) {
        const int ring = (int)(pk >> 16) - 1;
        const unsigned lstart = lcnt[ring];
        const int slot = lstart + (pk & 0xffffu);
        perm[slot] = (unsigned short)(it * 32 + lane);
        delta[slot] = __ldg(&row[ring]) - lstart;        // global offset of the chunk's ring group - its local start
      }
      total += __popc(__ballot_sync(0xffffffffu, pk != 0));
    }
    __syncwarp();
    // walk the chunk in ring order, four warp-rows at a time so that four point gathers are in flight per lane
    for (int t0 = 0; t0 < total; t0 += 128) {
      float4 p[4];
      int li[4];
      unsigned dl[4];
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const int t = t0 + j * 32 + lane;
        li[j] = t < total ? perm[t] : 0;
        dl[j] = t < total ? delta[t] : 0;
      }
#pragma unroll
      for (int j = 0; j < 4; j++) p[j] = __ldg(&buf.in[g0 + li[j]]);
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const int t = t0 + j * 32 + lane;
        if (t < total) {
          const unsigned dst = gb + dl[j] + (unsigned)t;
          buf.bpt[dst] = make_float4(p[j].x, p[j].y, p[j].z, __int_as_float(chunk * kChunk + li[j]));
          // (azimuth, input index) in bucket order: all k_sort_rings reads
          if (prm.want_order) buf.baz[dst] = make_uint2(fbits(buf.az[g0 + li[j]]), (unsigned)(chunk * kChunk + li[j]));
        }
      }
    }
  }
  __syncthreads();                                                // s_sbase is complete
  if (live) {
    // sector records (r, z, input index), four coalesced point loads in flight per lane
#pragma unroll
    for (int h = 0; h < kChunk / 32 / 4; h++) {
      float4 p[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int li = (h * 4 + u) * 32 + lane;
        p[u] = spack[h * 4 + u] ? __ldg(&buf.in[g0 + li]) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const unsigned sp = spack[h * 4 + u];
        if (sp) {
          const int sec = (int)(sp >> 16) - 1;
          const int i = chunk * kChunk + (h * 4 + u) * 32 + lane;
          buf.spt[gb + (unsigned)(s_sbase[sec] + (int)(sp & 0xffffu))] = make_float4(star_radius(p[u].x, p[u].y), p[u].z, __int_as_float(i), 0.f);
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Star-shaped search, sort by planar radius (star_shaped_search.cpp:109). Order: (r, input index) — the reference's
// introsort order for equal r is unspecified; ties raise F_TIE_SECTOR.
//
// Register-resident bitonic network: thread t owns elements t*EPL .. t*EPL+EPL-1 (32-bit radius bits + the element's slot
// in the unsorted sector as payload). Strides below EPL are register-only compare-exchanges, strides below 32*EPL go
// through warp shuffles, larger strides (multi-warp CTAs only) exchange through shared memory. One warp sorts up to 1024
// points (k_star_sort_warp, one 32-thread CTA per sector so that all control flow around the shuffles is provably
// uniform), eight warps up to 8192 (k_star_sort_big / k_star_refine, work lists). Returns true when two points share a
// radius: their order is what the reference's std::sort leaves (urf_stdsort.cuh), which the network does not see — such a
// sector, like any sector beyond 8192 points, is redone by slow_sort_sector.
constexpr int kWarpCap = 1024, kCtaCap = 8192;

// LIST (single-warp only): the n elements to sort are given as (radius bits, slot in src) pairs in s_xk / s_xe instead of
// being all of src[0 .. n) — the near-first prefix of k_star_sort_warp.
template <int EPL, int WARPS, bool LIST = false>
__device__ __forceinline__ bool bitonic_sector(const float4* __restrict__ src, float4* __restrict__ dst, int n, int tid,
                                               unsigned* s_xk, unsigned* s_xe) {
  constexpr int THREADS = WARPS * 32;                // sorts up to THREADS * EPL elements
  // LIST with WARPS > 1: the list lives in the exchange buffers; every thread has taken its entries into registers before
  // the barrier in front of the first cross-warp exchange lets anybody overwrite them
  const int lane = tid & 31;
  unsigned key[EPL], el[EPL];
#pragma unroll
  for (int r = 0; r < EPL; r++) {
    const int e = tid * EPL + r;
    key[r] = 0xffffffffu; el[r] = 0u;
    if (e < n) {
      if (LIST) { key[r] = s_xk[e]; el[r] = s_xe[e]; }
      else { key[r] = fbits(src[e].x); el[r] = (unsigned)e; }
    }
  }
  // intra-thread compare-exchange network for strides EPL/2 .. 1 of merge phase k (compile-time register indices)
  auto intra = [&](int k_over_epl, auto kc) {
    constexpr int K = decltype(kc)::value;             // K > 0: merge phase k = K < EPL (direction depends on r only)
#pragma unroll
    for (int j = (K > 0 ? K : EPL) >> 1; j > 0; j >>= 1) {
#pragma unroll
      for (int r = 0; r < EPL; r++) {
        if ((r & j) == 0) {
          const bool asc = K > 0 ? ((r & K) == 0) : ((tid & k_over_epl) == 0);
          const bool sw = (key[r] > key[r | j]) == asc;
          const unsigned ka = sw ? key[r | j] : key[r], kb = sw ? key[r] : key[r | j];
          const unsigned ea = sw ? el[r | j] : el[r], eb = sw ? el[r] : el[r | j];
          key[r] = ka; key[r | j] = kb; el[r] = ea; el[r | j] = eb;
        }
      }
    }
  };
  // phases k = 2 .. EPL/2: entirely inside the thread
  if (EPL > 2) intra(0, std::integral_constant<int, 2>());
  if (EPL > 4) intra(0, std::integral_constant<int, 4>());
  if (EPL > 8) intra(0, std::integral_constant<int, 8>());
  if (EPL > 16) intra(0, std::integral_constant<int, 16>());
  // phases k = EPL .. N: thread-level strides (shuffles / shared memory, runtime loop), then the intra-thread strides
  for (int ke = 1; ke <= THREADS; ke <<= 1) {          // ke = k / EPL
    for (int tj = ke >> 1; tj > 0; tj >>= 1) {         // partner thread = tid ^ tj
      const bool keep_min = ((tid & tj) == 0) == ((tid & ke) == 0);
      if (tj < 32) {
#pragma unroll
        for (int r = 0; r < EPL; r++) {
          const unsigned o = __shfl_xor_sync(0xffffffffu, key[r], tj);
          const unsigned oe = __shfl_xor_sync(0xffffffffu, el[r], tj);
          const bool take = (o < key[r]) == keep_min;            // branch-free; taking an equal key is harmless
          key[r] = take ? o : key[r];
          el[r] = take ? oe : el[r];
        }
      } else {                                         // partner in another warp: exchange through shared memory
        __syncthreads();
#pragma unroll
        for (int r = 0; r < EPL; r++) { s_xk[r * THREADS + tid] = key[r]; s_xe[r * THREADS + tid] = el[r]; }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < EPL; r++) {
          const unsigned o = s_xk[r * THREADS + (tid ^ tj)], oe = s_xe[r * THREADS + (tid ^ tj)];
          const bool take = (o < key[r]) == keep_min;
          key[r] = take ? o : key[r];
          el[r] = take ? oe : el[r];
        }
      }
    }
    intra(ke, std::integral_constant<int, 0>());
  }
  // write out + tie detection against the predecessor in sorted order
  unsigned prev0 = __shfl_up_sync(0xffffffffu, key[EPL - 1], 1);
  if (WARPS > 1) {
    __syncthreads();
    if (lane == 31) s_xk[tid >> 5] = key[EPL - 1];
    __syncthreads();
    if (lane == 0 && tid > 0) prev0 = s_xk[(tid >> 5) - 1];
  }
  bool tie = false;
#pragma unroll
  for (int r = 0; r < EPL; r++) {
    const int e = tid * EPL + r;
    const unsigned prev = r > 0 ? key[r - 1] : prev0;
    if (e < n) {
      dst[e] = src[el[r]];
      if (e > 0 && prev == key[r]) tie = true;
    }
  }
  return tie;
}

// whole sector of up to kWarpCap points by one warp; true = radius tie
__device__ __forceinline__ bool sort_sector_warp(const float4* __restrict__ src, float4* __restrict__ dst, int n, int lane) {
  if (n <= 128) return bitonic_sector<4, 1>(src, dst, n, lane, nullptr, nullptr);
  if (n <= 256) return bitonic_sector<8, 1>(src, dst, n, lane, nullptr, nullptr);
  if (n <= 512) return bitonic_sector<16, 1>(src, dst, n, lane, nullptr, nullptr);
  return bitonic_sector<32, 1>(src, dst, n, lane, nullptr, nullptr);
}

// Near-first selection (see k_star_sort_warp): all radius loads of the sector are issued together, the pivot is the 18th
// smallest of 32 evenly spaced samples, and the (radius bits, slot) pairs below the pivot are appended to the shared
// lists in any order. Returns their number.
template <int EPL>
__device__ __forceinline__ int select_near(const float4* __restrict__ src, int n, int lane, unsigned* s_pk, unsigned* s_pe, int pivot_rank, int cap = kWarpCap) {
  const unsigned mine = fbits(src[(int)(((unsigned)lane * (unsigned)n) >> 5)].x);
  unsigned key[EPL];
#pragma unroll
  for (int r = 0; r < EPL; r++) {
    const int e = r * 32 + lane;
    key[r] = e < n ? fbits(src[e].x) : 0xffffffffu;
  }
  int rank = 0;                                        // ranks of the samples are a permutation (ties broken by lane)
#pragma unroll
  for (int j = 0; j < 32; j++) { const unsigned o = __shfl_sync(0xffffffffu, mine, j); rank += (o < mine) || (o == mine && j < lane); }
  const unsigned pivot = __shfl_sync(0xffffffffu, mine, __ffs(__ballot_sync(0xffffffffu, rank == pivot_rank)) - 1);
  const unsigned lt = (1u << lane) - 1u;
  int m = 0;
#pragma unroll
  for (int r = 0; r < EPL; r++) {
    const bool sel = key[r] < pivot;                   // padding keys are 0xffffffff: never selected
    const unsigned bs = __ballot_sync(0xffffffffu, sel);
    const int pos = m + __popc(bs & lt);
    if (sel && pos < cap) { s_pk[pos] = key[r]; s_pe[pos] = (unsigned)(r * 32 + lane); }   // beyond cap: counted only
    m += __popc(bs);
  }
  __syncwarp();
  return m;
}

// The other side of a near-first split, for k_star_refine: the (radius bits, slot) pairs of the points whose radius lies
// ABOVE `kmax` (the largest radius of the sorted prefix; prefix radii are all below the pivot, the rest at or above it),
// appended to the shared lists in any order. Returns their number.
template <int EPL>
__device__ __forceinline__ int select_far(const float4* __restrict__ src, int n, int lane, unsigned* s_pk, unsigned* s_pe, unsigned kmax) {
  unsigned key[EPL];
#pragma unroll
  for (int r = 0; r < EPL; r++) {
    const int e = r * 32 + lane;
    key[r] = e < n ? fbits(src[e].x) : 0u;             // padding: radius bits 0 are never above kmax
  }
  const unsigned lt = (1u << lane) - 1u;
  int m = 0;
#pragma unroll
  for (int r = 0; r < EPL; r++) {
    const bool sel = key[r] > kmax;
    const unsigned bs = __ballot_sync(0xffffffffu, sel);
    if (sel) { const int pos = m + __popc(bs & lt); s_pk[pos] = key[r]; s_pe[pos] = (unsigned)(r * 32 + lane); }
    m += __popc(bs);
  }
  __syncwarp();
  return m;
}

// One 32-thread CTA per sector: sector index and size derive from blockIdx, so the compiler knows the control flow
// around the shuffles is warp-uniform (no convergence barriers around every SHFL).
//
// Near-first sort. The edge search (k_star_scan) walks a sector outwards and stops at its first edge point, so the far
// part of a sector is usually never looked at. Sectors above kPrefixMin points are therefore split at a pivot radius (the
// 18th smallest of 32 evenly spaced samples): points below the pivot are compacted into shared memory and sorted (about
// half the sector -> a network of half the width, ~40 % of the compare-exchanges); the rest is not written at all.
// tab.sorted_len tells k_star_scan how far it may walk; a sector whose walk reaches the end of the sorted prefix
// without an edge is put on tab.refine and redone in full (k_star_refine: full sort + star_resume_walk). Exact either
// way: every point of the prefix is closer than every point behind it.
constexpr int kPrefixMin = 128;
// Sorts of more than 512 elements go to k_star_sort_big's list, which leaves this kernel with the networks of up to 16
// elements per lane (64 registers, 32 resident warps per SM to hide the shuffle latency; measured and dropped: networks
// of up to 32 elements per lane here, 128 registers and 16 warps per SM, 2 % slower per step at C2 x 128). (Also measured
// and dropped: a keys-only network — one SHFL + two VIMNMX per remote compare-exchange instead of two SHFL, a compare and
// two selects — with the payload recovered by a binary search of every key in the sorted keys: 30 % fewer instructions,
// but 0.7 % slower per step.)
__global__ void __launch_bounds__(32, 32) k_star_sort_warp(DevBuffers buf, DevParams prm, int S) {
  constexpr int kList = 32 * 16;                                        // longest list this kernel sorts itself
  __shared__ unsigned s_pk[kList], s_pe[kList];
  const int b = blockIdx.y, s = blockIdx.x, lane = threadIdx.x;
  ScanTab& tab = buf.tab[b];
  const int base = tab.sect_start[s], n = tab.sect_start[s + 1] - base;
  if (lane == 0) tab.sorted_len[s] = n;
  if (n <= 0) return;
  const float4* src = buf.spt + (size_t)b * S + base;
  float4* dst = buf.ssorted + (size_t)b * S + base;
  if (n == 1) { if (lane == 0) dst[0] = src[0]; return; }
  if (n > kWarpCap) {                                                   // hand over to the CTA sort / the fallback
    if (lane == 0) {
      if (n <= kCtaCap) tab.biglist[atomicAdd(&tab.nbig, 1)] = (unsigned short)s;
      else tab.slowlist[atomicAdd(&tab.nslow, 1)] = (unsigned short)s;
    }
    return;
  }
  bool tie;
  int m = 0;
  if (prm.star_prefix && n > kPrefixMin) {
    if (n <= 256) m = select_near<8>(src, n, lane, s_pk, s_pe, kStarPivot, kList);
    else if (n <= 512) m = select_near<16>(src, n, lane, s_pk, s_pe, kStarPivot, kList);
    else m = select_near<32>(src, n, lane, s_pk, s_pe, kStarPivot, kList);
  }
  const bool near = m >= 32 && 4 * m <= 3 * n;                          // worth it: sort the near part only
  if ((near ? m : n) > kList) {                                         // a wide network: eight warps do it (k_star_sort_big)
    if (lane == 0) tab.biglist[atomicAdd(&tab.nbig, 1)] = (unsigned short)s;
    return;
  }
  if (near) {
    if (m <= 128) tie = bitonic_sector<4, 1, true>(src, dst, m, lane, s_pk, s_pe);
    else if (m <= 256) tie = bitonic_sector<8, 1, true>(src, dst, m, lane, s_pk, s_pe);
    else tie = bitonic_sector<16, 1, true>(src, dst, m, lane, s_pk, s_pe);
    if (lane == 0) tab.sorted_len[s] = m;
  } else {
    if (n <= 128) tie = bitonic_sector<4, 1>(src, dst, n, lane, nullptr, nullptr);
    else if (n <= 256) tie = bitonic_sector<8, 1>(src, dst, n, lane, nullptr, nullptr);
    else tie = bitonic_sector<16, 1>(src, dst, n, lane, nullptr, nullptr);
  }
  if (__any_sync(0xffffffffu, tie) && lane == 0) tab.slowlist[atomicAdd(&tab.nslow, 1)] = (unsigned short)s;   // sets F_TIE_SECTOR there
}

// Exact fallback sort of one sector by all threads of the CTA (bitonic; shared memory up to `cap` keys, global scratch
// beyond): sectors larger than kCtaCap and sectors holding EQUAL radii. Keys are (radius bits, input index). Without equal
// radii any correct sort gives the reference's order. With them (F_TIE_SECTOR) the reference's order is what libstdc++'s
// introsort leaves when it sorts the sector's points in push_back (= input) order by radius alone
// (star_shaped_search.cpp:109): the points are put back into input order (second bitonic pass, keyed by index) and ONE
// thread runs the restated std::sort (urf_stdsort.cuh) over them.
__device__ void slow_sort_sector(const DevBuffers& buf, int b, int S, int base, int n, unsigned long long* s_keys, int cap) {
  const float4* src = buf.spt + (size_t)b * S + base;
  float4* dst = buf.ssorted + (size_t)b * S + base;
  const int npad = next_pow2(n < 2 ? 2 : n);
  unsigned long long* keys = npad <= cap ? s_keys : buf.sortbuf + 2 * ((size_t)b * S + base);
  __syncthreads();
  for (int t = threadIdx.x; t < npad; t += blockDim.x)
    keys[t] = t < n ? (((unsigned long long)fbits(src[t].x) << 32) | (unsigned)__float_as_int(src[t].z)) : ~0ull;
  __syncthreads();
  cta_bitonic(keys, npad);
  bool tie = false;
  for (int t = threadIdx.x + 1; t < n; t += blockDim.x) if ((unsigned)(keys[t - 1] >> 32) == (unsigned)(keys[t] >> 32)) tie = true;
  if (__syncthreads_or(tie)) {                           // uniform: reproduce std::sort's order of the equal radii
    for (int t = threadIdx.x; t < n; t += blockDim.x) { const unsigned long long k = keys[t]; keys[t] = (k << 32) | (k >> 32); }
    __syncthreads();
    cta_bitonic(keys, npad);                             // ascending input index = push_back order (padding keys stay last)
    for (int t = threadIdx.x; t < n; t += blockDim.x) { const unsigned long long k = keys[t]; keys[t] = (k << 32) | (k >> 32); }
    __syncthreads();
    if (threadIdx.x == 0) { urfsort::std_sort(keys, n); atomicOr(&buf.out[b].flags, F_TIE_SECTOR); }
    __syncthreads();
  }
  // rebuild the records in key order (z comes from the input record of that index)
  for (int t = threadIdx.x; t < n; t += blockDim.x) {
    const unsigned long long k = keys[t];
    const int idx = (int)(unsigned)k;
    dst[t] = make_float4(bitsf((unsigned)(k >> 32)), buf.in[(size_t)b * S + idx].z, __int_as_float(idx), 0.f);
  }
  __syncthreads();
}

// Near-first selection for the eight-warp sort (see k_star_sort_warp): pivot = the 144th smallest of 256 evenly spaced
// samples (56 %), the (radius bits, slot) pairs below it appended to the shared lists in any order. Returns their number.
template <int EPL>
__device__ __forceinline__ int select_near_cta(const float4* __restrict__ src, int n, int tid, unsigned* s_pk, unsigned* s_pe, unsigned* s_misc, int pivot_rank) {
  const unsigned mine = fbits(src[(int)(((unsigned)tid * (unsigned)n) >> 8)].x);
  unsigned key[EPL];
#pragma unroll
  for (int r = 0; r < EPL; r++) {
    const int e = r * 256 + tid;
    key[r] = e < n ? fbits(src[e].x) : 0xffffffffu;
  }
  __syncthreads();                                     // the lists are free (previous sector done)
  s_pk[tid] = mine;
  if (tid == 0) s_misc[1] = 0u;
  __syncthreads();
  int rank = 0;                                        // ranks of the samples are a permutation (ties broken by thread)
  for (int j = 0; j < 256; j++) { const unsigned o = s_pk[j]; rank += (o < mine) || (o == mine && j < tid); }
  if (rank == pivot_rank) s_misc[0] = mine;
  __syncthreads();
  const unsigned pivot = s_misc[0];
  __syncthreads();                                     // everybody has read the samples: the lists may be overwritten
  const unsigned lt = (1u << (tid & 31)) - 1u;
#pragma unroll
  for (int r = 0; r < EPL; r++) {
    const bool sel = key[r] < pivot;                   // padding keys are 0xffffffff: never selected
    const unsigned bs = __ballot_sync(0xffffffffu, sel);
    unsigned wb = 0;
    if ((tid & 31) == 0 && bs) wb = atomicAdd(&s_misc[1], (unsigned)__popc(bs));
    wb = __shfl_sync(0xffffffffu, wb, 0);
    if (sel) { const unsigned pos = wb + __popc(bs & lt); s_pk[pos] = key[r]; s_pe[pos] = (unsigned)(r * 256 + tid); }
  }
  __syncthreads();
  return (int)s_misc[1];
}

// eight-warp register network on a whole sector (LIST = false) or on the m listed elements (LIST = true); true = radius tie
template <bool LIST>
__device__ __forceinline__ bool sort_sector_cta(const float4* __restrict__ src, float4* __restrict__ dst, int n, int tid, unsigned* s_xk, unsigned* s_xe) {
  if (n <= 1024) return bitonic_sector<4, 8, LIST>(src, dst, n, tid, s_xk, s_xe);
  if (n <= 2048) return bitonic_sector<8, 8, LIST>(src, dst, n, tid, s_xk, s_xe);
  if (n <= 4096) return bitonic_sector<16, 8, LIST>(src, dst, n, tid, s_xk, s_xe);
  return bitonic_sector<32, 8, LIST>(src, dst, n, tid, s_xk, s_xe);
}

// k_star_sort_big: the sectors k_star_sort_warp handed over. tab.biglist (1025 .. kCtaCap points): eight-warp register
// network, near-first like the single-warp sort (only the points below a sampled pivot radius are sorted, sorted_len tells
// k_star_scan how far it may walk), redone at once in full by the exact fallback when it meets equal radii; tab.slowlist
// (larger sectors, and sectors in which the single-warp sort met equal radii): exact fallback, whole sector.
constexpr size_t kStarCtaSmem = 2 * sizeof(unsigned) * kCtaCap;            // 64 KB: exchange buffers / 8192 64-bit keys
__global__ void __launch_bounds__(256) k_star_sort_big(DevBuffers buf, DevParams prm, int S) {
  extern __shared__ unsigned s_dyn[];
  const int b = blockIdx.y;
  ScanTab& tab = buf.tab[b];
  unsigned* s_xk = s_dyn;
  unsigned* s_xe = s_dyn + kCtaCap;
  __shared__ int s_tie;
  __shared__ unsigned s_misc[2];
  const int nbig = tab.nbig, nslow = tab.nslow;
  for (int w = blockIdx.x; w < nbig; w += gridDim.x) {
    const int s = tab.biglist[w];
    const int base = tab.sect_start[s], n = tab.sect_start[s + 1] - base;
    const float4* src = buf.spt + (size_t)b * S + base;
    float4* dst = buf.ssorted + (size_t)b * S + base;
    if (threadIdx.x == 0) s_tie = 0;
    int m = 0;
    if (prm.star_prefix) {
      if (n <= 2048) m = select_near_cta<8>(src, n, threadIdx.x, s_xk, s_xe, s_misc, 8 * kStarPivot + 7);
      else if (n <= 4096) m = select_near_cta<16>(src, n, threadIdx.x, s_xk, s_xe, s_misc, 8 * kStarPivot + 7);
      else m = select_near_cta<32>(src, n, threadIdx.x, s_xk, s_xe, s_misc, 8 * kStarPivot + 7);
    }
    const bool near = m >= 256 && 4 * m <= 3 * n;                          // uniform: m comes from shared memory
    const bool tie = near ? sort_sector_cta<true>(src, dst, m, threadIdx.x, s_xk, s_xe) : sort_sector_cta<false>(src, dst, n, threadIdx.x, s_xk, s_xe);
    if (near && threadIdx.x == 0) tab.sorted_len[s] = m;
    __syncthreads();
    if (tie) s_tie = 1;
    __syncthreads();
    const bool redo = s_tie != 0;
    __syncthreads();
    if (redo) {
      if (threadIdx.x == 0) tab.sorted_len[s] = n;
      slow_sort_sector(buf, b, S, base, n, reinterpret_cast<unsigned long long*>(s_dyn), kCtaCap);
    }
  }
  for (int w = blockIdx.x; w < nslow; w += gridDim.x) {
    const int s = tab.slowlist[w];
    const int base = tab.sect_start[s], n = tab.sect_start[s + 1] - base;
    if (threadIdx.x == 0) tab.sorted_len[s] = n;
    slow_sort_sector(buf, b, S, base, n, reinterpret_cast<unsigned long long*>(s_dyn), kCtaCap);
  }
}

// the exact fallback sort (see slow_sort_sector) by ONE warp, for a sector of up to kWarpCap points: keys in the warp's own
// shared memory, warp barriers only
__device__ __forceinline__ void warp_bitonic(unsigned long long* keys, int npad, int lane) {
  for (int k = 2; k <= npad; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = lane; t < (npad >> 1); t += 32) {
        const int i = 2 * t - (t & (j - 1)), l = i + j;
        const bool up = (i & k) == 0;
        const unsigned long long x = keys[i], y = keys[l];
        if ((x > y) == up) { keys[i] = y; keys[l] = x; }
      }
      __syncwarp();
    }
  }
}
__device__ void slow_sort_sector_warp(const DevBuffers& buf, int b, int S, int base, int n, unsigned long long* keys, int lane) {
  const float4* src = buf.spt + (size_t)b * S + base;
  float4* dst = buf.ssorted + (size_t)b * S + base;
  const int npad = next_pow2(n < 2 ? 2 : n);
  for (int t = lane; t < npad; t += 32)
    keys[t] = t < n ? (((unsigned long long)fbits(src[t].x) << 32) | (unsigned)__float_as_int(src[t].z)) : ~0ull;
  __syncwarp();
  warp_bitonic(keys, npad, lane);
  bool tie = false;
  for (int t = lane + 1; t < n; t += 32) if ((unsigned)(keys[t - 1] >> 32) == (unsigned)(keys[t] >> 32)) tie = true;
  if (__any_sync(0xffffffffu, tie)) {                    // reproduce std::sort's order of the equal radii (see slow_sort_sector)
    for (int t = lane; t < n; t += 32) { const unsigned long long k = keys[t]; keys[t] = (k << 32) | (k >> 32); }
    __syncwarp();
    warp_bitonic(keys, npad, lane);
    for (int t = lane; t < n; t += 32) { const unsigned long long k = keys[t]; keys[t] = (k << 32) | (k >> 32); }
    __syncwarp();
    if (lane == 0) { urfsort::std_sort(keys, n); atomicOr(&buf.out[b].flags, F_TIE_SECTOR); }
    __syncwarp();
  }
  for (int t = lane; t < n; t += 32) {
    const unsigned long long k = keys[t];
    const int idx = (int)(unsigned)k;
    dst[t] = make_float4(bitsf((unsigned)(k >> 32)), buf.in[(size_t)b * S + idx].z, __int_as_float(idx), 0.f);
  }
  __syncwarp();
}

// resumed walk of a refined sector (entry w of tab.refine) over its completely sorted points, by one thread
__device__ void star_resume_walk(const DevBuffers& buf, const DevParams& prm, ScanTab& tab, int b, int S, int w, int s, const float4* dst, int n) {
  tab.sorted_len[s] = n;
  StarState st;
  st.avg = tab.resume[w][0]; st.dev = tab.resume[w][1]; st.nan = tab.resume[w][2];
  int i = __float_as_int(tab.resume[w][3]);            // >= 32: a prefix is never shorter
  const float4 last = dst[i - 1];
  st.bx = last.x; st.by = last.y;
  int hit = -1;
  while (i < n && hit < 0) {
    float4 p[4];
#pragma unroll
    for (int u = 0; u < 4; u++) p[u] = dst[min(i + u, n - 1)];
#pragma unroll
    for (int u = 0; u < 4; u++)
      if (hit < 0 && i + u < n && star_step(prm, st, i + u, p[u].x, p[u].y)) hit = i + u;
    i += 4;
  }
  if (hit >= 0) curb_hit(buf, prm, b, scan_base(b, S), __float_as_int(dst[hit].z), -1);     // star_shaped_search.cpp:146
}

// the same by one WARP (all 32 lanes call it): per tile of 32 points every lane computes what does not depend on the
// recurrence for one point (slope, radius step, 1 / i: the IEEE divisions), then all lanes run the dependent part of the
// 32 points in lock step on their own copy of the state (values handed round by shuffles), so control flow stays uniform.
__device__ __forceinline__ void star_resume_walk_warp(const DevBuffers& buf, const DevParams& prm, ScanTab& tab, int b, int S, int w, int s,
                                                      const float4* dst, int n, int lane) {
  if (lane == 0) tab.sorted_len[s] = n;
  StarState st;
  st.avg = tab.resume[w][0]; st.dev = tab.resume[w][1]; st.nan = tab.resume[w][2];
  const int n0 = __float_as_int(tab.resume[w][3]);     // >= 32: a prefix is never shorter
  st.bx = 0.f; st.by = 0.f;                            // unused: slopes come from the points themselves
  int hit = -1;
  for (int t0 = n0; t0 < n && hit < 0; t0 += 32) {
    const int e = min(t0 + lane, n - 1);
    const float4 p = dst[e], pp = dst[e - 1];
    float dx;
    const float slp = star_slope(pp.x, pp.y, p.x, p.y, &dx);
    const float dxk = __fmul_rn(dx, prm.kdist);
    const float inv = star_inv(e);
    const int cnt = min(32, n - t0);
    for (int j = 0; j < cnt; j++) {
      const float sj = __shfl_sync(0xffffffffu, slp, j), dj = __shfl_sync(0xffffffffu, dxk, j), ij = __shfl_sync(0xffffffffu, inv, j);
      if (star_update(prm, st, t0 + j, sj, dj, ij)) { hit = t0 + j; break; }
    }
  }
  if (hit >= 0 && lane == 0) curb_hit(buf, prm, b, scan_base(b, S), __float_as_int(dst[hit].z), -1);   // star_shaped_search.cpp:146
}

// k_star_refine: second pass for the sectors whose edge search ran off their sorted prefix (tab.refine, filled by
// k_star_scan): the rest of the sector is sorted behind the prefix (single-warp path; the CTA path sorts the whole sector
// again), then one thread resumes the walk at point n0 with the saved running mean / deviation — the first n0 points of
// the full order are the prefix already walked (all of them are closer than the rest). Sectors of up to kWarpCap points:
// one WARP per sector (register network, exact fallback on equal radii in the warp's shared memory), the eight warps of a
// CTA working on eight sectors; larger sectors: the whole CTA, one at a time.
__global__ void __launch_bounds__(256) k_star_refine(DevBuffers buf, DevParams prm, int S) {
  extern __shared__ unsigned s_dyn[];
  const int b = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  ScanTab& tab = buf.tab[b];
  __shared__ int s_tie;
  const int nref = tab.nrefine;
  unsigned long long* wkeys = reinterpret_cast<unsigned long long*>(s_dyn) + (size_t)warp * kWarpCap;   // 8 x 8 KB
  for (int w = blockIdx.x * 8 + warp; w < nref; w += gridDim.x * 8) {
    const int s = tab.refine[w];
    const int base = tab.sect_start[s], n = tab.sect_start[s + 1] - base;
    if (n > kWarpCap) continue;                                            // second loop
    const float4* src = buf.spt + (size_t)b * S + base;
    float4* dst = buf.ssorted + (size_t)b * S + base;
    // dst[0, n0) already holds the n0 closest points in order (the walked prefix): only the rest is sorted, behind it
    const int n0 = __float_as_int(tab.resume[w][3]);
    unsigned* s_pk = reinterpret_cast<unsigned*>(wkeys);
    unsigned* s_pe = s_pk + kWarpCap;
    const unsigned kmax = fbits(dst[n0 - 1].x);
    int m;
    if (n <= 256) m = select_far<8>(src, n, lane, s_pk, s_pe, kmax);
    else if (n <= 512) m = select_far<16>(src, n, lane, s_pk, s_pe, kmax);
    else m = select_far<32>(src, n, lane, s_pk, s_pe, kmax);
    bool tie;
    if (m != n - n0) tie = true;                                           // cannot happen (prefix = everything below the pivot); exact path if it does
    else if (m <= 128) tie = bitonic_sector<4, 1, true>(src, dst + n0, m, lane, s_pk, s_pe);
    else if (m <= 256) tie = bitonic_sector<8, 1, true>(src, dst + n0, m, lane, s_pk, s_pe);
    else if (m <= 512) tie = bitonic_sector<16, 1, true>(src, dst + n0, m, lane, s_pk, s_pe);
    else tie = bitonic_sector<32, 1, true>(src, dst + n0, m, lane, s_pk, s_pe);
    __syncwarp();
    if (__any_sync(0xffffffffu, tie)) slow_sort_sector_warp(buf, b, S, base, n, wkeys, lane);   // equal radii: whole sector, std::sort's order
    __syncwarp();
    star_resume_walk_warp(buf, prm, tab, b, S, w, s, dst, n, lane);
    __syncwarp();
  }
  __syncthreads();
  unsigned* s_xk = s_dyn;
  unsigned* s_xe = s_dyn + kCtaCap;
  for (int w = blockIdx.x; w < nref; w += gridDim.x) {
    const int s = tab.refine[w];
    const int base = tab.sect_start[s], n = tab.sect_start[s + 1] - base;
    if (n <= kWarpCap) continue;                                           // done above
    const float4* src = buf.spt + (size_t)b * S + base;
    float4* dst = buf.ssorted + (size_t)b * S + base;
    if (tid == 0) s_tie = 0;
    __syncthreads();
    bool tie = n <= kCtaCap ? sort_sector_cta<false>(src, dst, n, tid, s_xk, s_xe) : true;   // beyond the register networks: exact fallback
    if (tie) s_tie = 1;
    __syncthreads();
    if (s_tie) slow_sort_sector(buf, b, S, base, n, reinterpret_cast<unsigned long long*>(s_dyn), kCtaCap);
    __syncthreads();
    if (tid == 0) star_resume_walk(buf, prm, tab, b, S, w, s, dst, n);
    __syncthreads();
  }
}

// k_star_scan: one lane per sector walks its radius-sorted points with the reference's running mean / average absolute
// deviation recurrence (star_shaped_search.cpp:112-150) and marks the first edge point. Per 32-point tile the warp first
// computes, 32 points of one sector at a time, everything that does not depend on the recurrence (slope, radius step,
// 1 / i — including the IEEE divisions) into shared memory; the serial walk is then a dozen dependent float operations
// per point.
constexpr int kScanWarps = 2;
__global__ void __launch_bounds__(kScanWarps * 32) k_star_scan(DevBuffers buf, DevParams prm, int S) {
  const int b = blockIdx.y, warp = threadIdx.x >> 5, lane = lane_id();
  __shared__ float s_slp[kScanWarps][32][33];
  __shared__ float s_dxk[kScanWarps][32][33];
  __shared__ float s_inv[kScanWarps][32][33];
  ScanTab& tab = buf.tab[b];
  const int s = (blockIdx.x * kScanWarps + warp) * 32 + lane;
  int base = 0, n = 0, whole = 0;
  if (s < kSectKeys) {
    base = tab.sect_start[s]; whole = tab.sect_start[s + 1] - base;
    n = min(whole, tab.sorted_len[s]);               // walk the sorted prefix only
  }
  const float4* all = buf.ssorted + (size_t)b * S;
  StarState st;
  star_init(st, 0.f, 0.f);
  bool done = n <= 1;                                                   // star_shaped_search.cpp:112
  int hit = -1;
  int nmax = n;
  for (int o = 16; o > 0; o >>= 1) nmax = max(nmax, __shfl_xor_sync(0xffffffffu, nmax, o));
  for (int t0 = 0; t0 < nmax; t0 += 32) {
    // stage tile [t0, t0 + 32) of all 32 sector rows: 8 rows at a time so that the 16 loads of a group are in flight
    // together (one L2 round trip per group instead of one per row). (Measured and dropped: 16 rows at a time with 8-byte
    // loads and the predecessor taken from the left neighbour by shuffle — 0.102 instead of 0.068 ms at C2 x 128.)
    for (int q0 = 0; q0 < 32; q0 += 8) {
      float4 p[8], pp[8];
      bool ok[8];
#pragma unroll
      for (int u = 0; u < 8; u++) {
        const int q = q0 + u;
        const int qn = __shfl_sync(0xffffffffu, n, q), qbase = __shfl_sync(0xffffffffu, base, q);
        const int qdone = __shfl_sync(0xffffffffu, (int)done, q);
        const int e = t0 + lane;
        ok[u] = !qdone && e < qn && e >= 1;
        const int at = ok[u] ? qbase + e : 1;
        p[u] = all[at]; pp[u] = all[at - 1];
      }
#pragma unroll
      for (int u = 0; u < 8; u++) {
        if (ok[u]) {
          float dx;
          s_slp[warp][q0 + u][lane] = star_slope(pp[u].x, pp[u].y, p[u].x, p[u].y, &dx);
          s_dxk[warp][q0 + u][lane] = __fmul_rn(dx, prm.kdist);
          s_inv[warp][q0 + u][lane] = star_inv(t0 + lane);
        }
      }
    }
    __syncwarp();
    if (!done) {
      const int e1 = min(32, n - t0);
      for (int e = (t0 == 0 ? 1 : 0); e < e1; e++) {
        const int i = t0 + e;
        if (star_update(prm, st, i, s_slp[warp][lane][e], s_dxk[warp][lane][e], s_inv[warp][lane][e])) { hit = i; done = true; break; }
      }
      if (t0 + 32 >= n) done = true;
    }
    __syncwarp();
    if (__all_sync(0xffffffffu, done)) break;
  }
  if (hit >= 0) curb_hit(buf, prm, b, scan_base(b, S), __float_as_int(all[base + hit].z), -1);   // star_shaped_search.cpp:146
  else if (n < whole) {                               // ran off the sorted prefix: sort in full, k_star_refine continues from here
    const int w = atomicAdd(&tab.nrefine, 1);
    tab.refine[w] = (unsigned short)s;
    tab.resume[w][0] = st.avg; tab.resume[w][1] = st.dev; tab.resume[w][2] = st.nan; tab.resume[w][3] = __int_as_float(n);
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// k_ring_detect: one thread per ring-bucket position: the x-zero test for which this point is the middle point p2
// (x_zero_method.cpp:30-67), the z-zero test centred on it (z_zero_method.cpp:21-72), and the ring's largest planar range
// (maxDistance, lidar_segmentation.cpp:271-274, as the largest double sum — see planar_sum_bits). The CTA stages its 256
// bucket positions plus a halo of curb_points on each side in shared memory as three coordinate arrays (plain global
// reads when curb_points exceeds kHalo). Both detectors are a cheap height gate followed by an expensive angle test
// (four double square roots, a double divide, acosf); about one point in eight passes a gate, scattered over most warps,
// so every thread evaluates only the gates and the CTA compacts the survivors into a work list that full warps then run
// the angle tests over (x-zero items from thread 0 upwards, z-zero items from thread 255 downwards). Points found to be
// curb points are marked in input order and entered into the curb bins (curb_hit); nothing else is written per point.
// Runs for curb_points other than the default 5 (k_ring_detect4 below takes that), eight CTAs per SM (32 registers).
constexpr int kHalo = 32;
__global__ void __launch_bounds__(256, 8) k_ring_detect(DevBuffers buf, DevParams prm, int S) {
  const int b = blockIdx.y;
  const ScanOut& out = buf.out[b];
  const int p0 = blockIdx.x * 256, tid = threadIdx.x, p = p0 + tid;
  const unsigned gb = scan_base(b, S);
  const float4* bucket = buf.bpt + gb;
  // inside the scan's slot whatever n_order is, so the load need not wait for it
  const float4 me0 = p < S ? bucket[p] : make_float4(0.f, 0.f, 0.f, 0.f);
  const int N = out.n_order;
  __shared__ float s_x[256 + 2 * kHalo], s_y[256 + 2 * kHalo], s_z[256 + 2 * kHalo];
  __shared__ int s_rs[kRingKeys + 2];                     // ring_start of the rings this CTA touches, indexed by ring - k_lo
  __shared__ int s_base[256];                             // ring_start of each thread's ring
  __shared__ unsigned short s_item[512];                  // x-zero work items grow from 0 up, z-zero items from 511 down
  __shared__ unsigned char s_hit[256];
  __shared__ int s_klo, s_nx, s_nz;
  if (p0 >= N) return;
  if (tid < 32) {                                         // rings are contiguous in bucket order: first .. last ring of the CTA
    const int k_lo = ring_of_position(out.ring_start, p0), k_hi = ring_of_position(out.ring_start, min(p0 + 255, N - 1));
    if (tid == 0) { s_klo = k_lo; s_nx = 0; s_nz = 0; }
    for (int t = tid; t <= k_hi - k_lo + 1; t += 32) s_rs[t] = out.ring_start[k_lo + t];
  }
  const bool tiled = prm.curbPoints <= kHalo;
  const bool act = p < N;
  const float4 me = act ? me0 : make_float4(0.f, 0.f, 0.f, 0.f);
  if (tiled) {                                            // one bucket record per thread + a halo record for the first 64 threads
    s_x[kHalo + tid] = me.x; s_y[kHalo + tid] = me.y; s_z[kHalo + tid] = me.z;
    if (tid < 2 * kHalo) {
      const int ph = tid < kHalo ? p0 - kHalo + tid : p0 + 256 + tid - kHalo;
      const int sh = tid < kHalo ? tid : 256 + tid;
      if (ph >= 0 && ph < N) { const float4 h = bucket[ph]; s_x[sh] = h.x; s_y[sh] = h.y; s_z[sh] = h.z; }
    }
    s_hit[tid] = 0;
  }
  __syncthreads();
  int k = -1;
  bool hit = false, need_x = false, need_z = false;
  if (act) {
    int r = 0;
    while (p >= s_rs[r + 1]) r++;                         // p < N = the last staged entry at the latest
    k = s_klo + r;
    const int base = s_rs[r], n = s_rs[r + 1] - base, m = p - base;
    if (tiled) {
      s_base[tid] = base;
      const int off = base - (p0 - kHalo);                // ring-local index q lives at tile slot off + q
      const RingSoA ring{s_x + off, s_y + off, s_z + off};
      need_x = prm.x_zero && xzero_pre(prm, ring, n, m);
      need_z = prm.z_zero && zzero_pre_t<0>(prm, ring, n, m);
    } else {                                              // huge curb_points: straight from global memory
      const float4* ring = bucket + base;
      hit = (prm.x_zero && xzero_mark(prm, ring, n, m, buf.newY)) ||                  // x_zero_method.cpp:66
            (prm.z_zero && zzero_mark(prm, ring, n, m));                              // z_zero_method.cpp:71
    }
  }
  if (tiled) {
    const unsigned bx = __ballot_sync(0xffffffffu, need_x), bz = __ballot_sync(0xffffffffu, need_z);
    const unsigned lt = (1u << lane_id()) - 1u;
    int ox = 0, oz = 0;
    if (lane_id() == 0) {
      if (bx) ox = atomicAdd(&s_nx, __popc(bx));
      if (bz) oz = atomicAdd(&s_nz, __popc(bz));
    }
    ox = __shfl_sync(0xffffffffu, ox, 0); oz = __shfl_sync(0xffffffffu, oz, 0);
    if (need_x) s_item[ox + __popc(bx & lt)] = (unsigned short)tid;
    if (need_z) s_item[511 - (oz + __popc(bz & lt))] = (unsigned short)tid;
    __syncthreads();
    const int nx = s_nx, nz = s_nz;
    for (int it = tid; it < nx; it += 256) {                            // x-zero angle tests, x_zero_method.cpp:35-61
      const int t = s_item[it], base = s_base[t], off = base - (p0 - kHalo);
      const RingSoA ring{s_x + off, s_y + off, s_z + off};
      if (xzero_post(prm, ring, p0 + t - base, buf.newY)) s_hit[t] = 1;
    }
    for (int it = 255 - tid; it < nz; it += 256) {                      // z-zero angle tests, z_zero_method.cpp:23-66
      const int t = s_item[511 - it], base = s_base[t], off = base - (p0 - kHalo);
      const RingSoA ring{s_x + off, s_y + off, s_z + off};
      if (zzero_post_t<0>(prm, ring, p0 + t - base)) s_hit[t] = 1;
    }
    __syncthreads();
    hit = act && s_hit[tid];                                            // x_zero_method.cpp:66, z_zero_method.cpp:71
  }
  if (hit) curb_hit(buf, prm, b, gb, __float_as_int(me.w), k);
  // maxDistance[k], lidar_segmentation.cpp:271-274 (warp-aggregated when the whole warp sits in one ring)
  const unsigned long long sb = act ? planar_sum_bits(me.x, me.y) : 0ull;
  const int k0 = __shfl_sync(0xffffffffu, k, 0);
  if (__all_sync(0xffffffffu, k == k0)) {
    if (k0 >= 0) {
      const unsigned hi = (unsigned)(sb >> 32), mh = __reduce_max_sync(0xffffffffu, hi);
      const unsigned ml = __reduce_max_sync(0xffffffffu, hi == mh ? (unsigned)sb : 0u);
      if (lane_id() == 0) atomicMax(&buf.tab[b].maxs[k0], ((unsigned long long)mh << 32) | ml);   // result unused: a RED
    }
  } else if (act) atomicMax(&buf.tab[b].maxs[k], sb);
}

// k_ring_detect4: the same work for the default curb_points = 5 with FOUR consecutive bucket positions per thread (tile of
// 1024 positions + halo per CTA). The two height gates of a position only read z: of its own ring, 5 positions to either
// side (z-zero) and at -2 / +3 (x-zero). Four consecutive positions share a window of 14 heights, which the thread fetches
// with five 16-byte shared-memory loads instead of 4 x 14 scalar ones; ring lookup, work-list compaction and the maximum of
// the planar sums are amortised over the four positions as well. Same logic functions, same results as k_ring_detect.
// Six CTAs per SM (40 registers; measured 1.337 ms per step against 1.351 at five and 1.380 at four).
constexpr int kTile4 = 1024;
__global__ void __launch_bounds__(256, 6) k_ring_detect4(DevBuffers buf, DevParams prm, int S) {
  constexpr int CP = 5;
  const int b = blockIdx.y;
  const ScanOut& out = buf.out[b];
  const int p0 = blockIdx.x * kTile4, tid = threadIdx.x;
  const unsigned gb = scan_base(b, S);
  const float4* bucket = buf.bpt + gb;
  // inside the scan's slot whatever n_order is, so the loads need not wait for it
  float4 rec[4];
#pragma unroll
  for (int j = 0; j < 4; j++) { const int q = p0 + tid + 256 * j; rec[j] = q < S ? bucket[q] : make_float4(0.f, 0.f, 0.f, 0.f); }
  const int N = out.n_order;
  __shared__ __align__(16) float s_x[kTile4 + 2 * kHalo], s_y[kTile4 + 2 * kHalo], s_z[kTile4 + 2 * kHalo];
  __shared__ int s_rs[kRingKeys + 2];                     // ring_start of the rings this CTA touches, indexed by ring - k_lo
  __shared__ unsigned short s_itx[kTile4], s_itz[kTile4]; // x-zero / z-zero work items: tile positions that passed the gate
  __shared__ __align__(4) unsigned char s_hit[kTile4];
  __shared__ int s_klo, s_nx, s_nz;
  if (p0 >= N) return;
  if (tid < 32) {                                         // rings are contiguous in bucket order: first .. last ring of the CTA
    const int k_lo = ring_of_position(out.ring_start, p0), k_hi = ring_of_position(out.ring_start, min(p0 + kTile4 - 1, N - 1));
    if (tid == 0) { s_klo = k_lo; s_nx = 0; s_nz = 0; }
    for (int t = tid; t <= k_hi - k_lo + 1; t += 32) s_rs[t] = out.ring_start[k_lo + t];
  }
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const int t = tid + 256 * j;
    const bool in = p0 + t < N;
    s_x[kHalo + t] = in ? rec[j].x : 0.f; s_y[kHalo + t] = in ? rec[j].y : 0.f; s_z[kHalo + t] = in ? rec[j].z : 0.f;
    s_hit[t] = 0;
  }
  if (tid < 2 * kHalo) {
    const int ph = tid < kHalo ? p0 - kHalo + tid : p0 + kTile4 + tid - kHalo;
    const int sh = tid < kHalo ? tid : kTile4 + tid;
    float4 h = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ph >= 0 && ph < N) h = bucket[ph];
    s_x[sh] = h.x; s_y[sh] = h.y; s_z[sh] = h.z;
  }
  __syncthreads();
  // the thread's four consecutive positions t0 .. t0 + 3 of the tile; heights of tile slots t0 - 8 .. t0 + 11
  const int t0 = 4 * tid;
  float zw[20];
#pragma unroll
  for (int v = 0; v < 5; v++) {
    const float4 f = *reinterpret_cast<const float4*>(&s_z[kHalo + t0 - 8 + 4 * v]);
    zw[4 * v] = f.x; zw[4 * v + 1] = f.y; zw[4 * v + 2] = f.z; zw[4 * v + 3] = f.w;
  }
  const float4 fx = *reinterpret_cast<const float4*>(&s_x[kHalo + t0]), fy = *reinterpret_cast<const float4*>(&s_y[kHalo + t0]);
  const float xs[4] = {fx.x, fx.y, fx.z, fx.w}, ys[4] = {fy.x, fy.y, fy.z, fy.w};
  int r = 0;                                              // ring (relative to s_klo) of the current position
  unsigned nx_mask = 0, nz_mask = 0;
  unsigned long long smax = 0ull;                         // largest planar sum among the thread's positions of ring rmax
  int rmax = -1;
  const int kbase = s_klo;
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const int p = p0 + t0 + j;
    if (p >= N) break;
    while (p >= s_rs[r + 1]) r++;                         // p < N = the last staged entry at the latest
    const int base = s_rs[r], n = s_rs[r + 1] - base, m = p - base;
    const float z = zw[8 + j];
    // z-zero gate, zzero_pre_t<5> on the register window (z_zero_method.cpp:38-40,47-49,67-69)
    if (prm.z_zero && m >= CP && m <= (n - 1) - CP) {
      const float az0 = fabsf(z);
      float max1 = az0, max2 = az0;
#pragma unroll
      for (int u = 1; u <= CP; u++) { const float v = fabsf(zw[8 + j - u]); if (v > max1) max1 = v; }
#pragma unroll
      for (int u = 1; u <= CP; u++) { const float v = fabsf(zw[8 + j + u]); if (v > max2) max2 = v; }
      if ((__fsub_rn(max1, az0) >= prm.curbHeight || __fsub_rn(max2, az0) >= prm.curbHeight) && (double)fabsf(__fsub_rn(max1, max2)) >= 0.05)
        nz_mask |= 1u << j;
    }
    // x-zero gate, xzero_pre with this point as p2 = j + cp / 2 (x_zero_method.cpp:62-64)
    const int jx = m - CP / 2;
    if (prm.x_zero && jx >= CP && jx <= (n - 1) - CP) {
      const float za = zw[8 + j - CP / 2], zc = zw[8 + j - CP / 2 + CP];
      if ((fabsf(__fsub_rn(za, z)) >= prm.curbHeight || fabsf(__fsub_rn(zc, z)) >= prm.curbHeight) && (double)fabsf(__fsub_rn(za, zc)) >= 0.05)
        nx_mask |= 1u << j;
    }
    // maxDistance: the thread keeps the maximum for the ring of its last position; an earlier ring's goes out at once
    const unsigned long long sb = planar_sum_bits(xs[j], ys[j]);
    if (r != rmax) {
      if (rmax >= 0) atomicMax(&buf.tab[b].maxs[kbase + rmax], smax);
      rmax = r; smax = sb;
    } else if (sb > smax) smax = sb;
  }
  // compaction of the gate survivors into the two work lists (one shared counter bump per warp and list)
  {
    const int cx = __popc(nx_mask), cz = __popc(nz_mask);
    int px = cx, pz = cz;                                 // inclusive warp scans of the per-thread counts
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int ax = __shfl_up_sync(0xffffffffu, px, o), az = __shfl_up_sync(0xffffffffu, pz, o);
      if (lane_id() >= o) { px += ax; pz += az; }
    }
    int wx = 0, wz = 0;
    if (lane_id() == 31) { if (px) wx = atomicAdd(&s_nx, px); if (pz) wz = atomicAdd(&s_nz, pz); }
    wx = __shfl_sync(0xffffffffu, wx, 31); wz = __shfl_sync(0xffffffffu, wz, 31);
    int ox = wx + px - cx, oz = wz + pz - cz;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      if (nx_mask & (1u << j)) s_itx[ox++] = (unsigned short)(t0 + j);
      if (nz_mask & (1u << j)) s_itz[oz++] = (unsigned short)(t0 + j);
    }
  }
  // warp-level maximum of the planar sums when the whole warp ended in one ring, else one atomic per thread
  {
    const int r0 = __shfl_sync(0xffffffffu, rmax, 0);
    if (__all_sync(0xffffffffu, rmax == r0)) {
      if (r0 >= 0) {
        const unsigned hi = (unsigned)(smax >> 32), mh = __reduce_max_sync(0xffffffffu, hi);
        const unsigned ml = __reduce_max_sync(0xffffffffu, hi == mh ? (unsigned)smax : 0u);
        if (lane_id() == 0) atomicMax(&buf.tab[b].maxs[kbase + r0], ((unsigned long long)mh << 32) | ml);
      }
    } else if (rmax >= 0) atomicMax(&buf.tab[b].maxs[kbase + rmax], smax);
  }
  __syncthreads();
  const int nx = s_nx, nz = s_nz;
  auto ring_base = [&](int t) {                           // ring start of tile position t (a tile spans few rings)
    const int p = p0 + t;
    int a = 0;
    while (p >= s_rs[a + 1]) a++;
    return s_rs[a];
  };
  for (int it = tid; it < nx; it += 256) {                              // x-zero angle tests, x_zero_method.cpp:35-61
    const int t = s_itx[it];
    const int base = ring_base(t), off = base - (p0 - kHalo);
    const RingSoA ring{s_x + off, s_y + off, s_z + off};
    if (xzero_post(prm, ring, p0 + t - base, buf.newY)) s_hit[t] = 1;
  }
  for (int it = tid; it < nz; it += 256) {                              // z-zero angle tests, z_zero_method.cpp:23-66
    const int t = s_itz[it];
    const int base = ring_base(t), off = base - (p0 - kHalo);
    const RingSoA ring{s_x + off, s_y + off, s_z + off};
    if (zzero_post_t<CP>(prm, ring, p0 + t - base)) s_hit[t] = 1;
  }
  __syncthreads();
  const unsigned hits = *reinterpret_cast<const unsigned*>(&s_hit[t0]);  // x_zero_method.cpp:66, z_zero_method.cpp:71
  if (hits) {
    int rr = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int p = p0 + t0 + j;
      if (p >= N) break;
      while (p >= s_rs[rr + 1]) rr++;
      if ((hits >> (8 * j)) & 0xffu) curb_hit(buf, prm, b, gb, __float_as_int(bucket[p].w), kbase + rr);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// blindSpots as tables (urf_logic.cuh: CurbView, window_blocked, build_T_row, covered_T). Three short kernels — a cluster
// of eight CTAs per scan running the three phases behind cluster barriers was measured at 111 us against 71 us for the
// three launches (C2 x 128: the 722 window tests of a scan want more than eight CTAs' worth of warps at once).
// k_tab1: per scan — prefix counts of non-empty curb bins per ring, maxDistance / arc widths, q1..q4, reach := n_rings.
__global__ void __launch_bounds__(256) k_tab1(DevBuffers buf, DevParams prm) {
  const int b = blockIdx.y;
  const ScanOut& out = buf.out[b];
  ScanTab& tab = buf.tab[b];
  const int R = out.n_rings;
  const int warp = threadIdx.x >> 5, lane = lane_id();
  if (blockIdx.x == 0) for (int t = threadIdx.x; t < 2 * kDegBins; t += blockDim.x) tab.reach[t / kDegBins][t % kDegBins] = R;
  if (R <= 0) return;
  const size_t nb = (size_t)prm.channels * kDegBins;
  const unsigned* cmin = buf.cmin + (size_t)b * nb;
  unsigned short* ne = buf.ne + (size_t)b * prm.channels * (kDegBins + 1);
  for (int k = blockIdx.x * 8 + warp; k < R; k += gridDim.x * 8) {        // one warp per ring: 12 x 32 bins with a running carry
    unsigned carry = 0;
    for (int c = 0; c < (kDegBins + 31) / 32; c++) {
      const int bin = c * 32 + lane;
      const unsigned f = bin < kDegBins && cmin[(size_t)k * kDegBins + bin] != 0x7f800000u;
      const unsigned bal = __ballot_sync(0xffffffffu, f);
      if (bin < kDegBins) ne[(size_t)k * (kDegBins + 1) + bin] = (unsigned short)(carry + __popc(bal & ((1u << lane) - 1u)));
      carry += __popc(bal);
    }
    if (lane == 0) ne[(size_t)k * (kDegBins + 1) + kDegBins] = (unsigned short)carry;
  }
  if (blockIdx.x != 0) return;
  const float arc = arc_distance(prm, maxdist_from_bits(tab.maxs[0]));   // blind_spots.cpp:65
  for (int k = threadIdx.x; k < R; k += blockDim.x) {
    const float md = maxdist_from_bits(tab.maxs[k]);                     // lidar_segmentation.cpp:271-274
    tab.maxdist[k] = fbits(md);
    tab.A[k] = ring_width(arc, md);                                      // :142
  }
  if (threadIdx.x < 4) {
    CurbView cv{cmin, buf.cmax + (size_t)b * nb, ne};
    tab.q[threadIdx.x] = blind_quarter(prm, cv, R, threadIdx.x);         // :13-57 (reads the curb bins only)
  }
}

// k_reach: one warp per (direction, window start i): lanes test 32 rings at a time whether ring k holds a curb point
// inside window i and stop at the first blocked ring — reach[dir][i] (blind_spots.cpp:107-171 / :216-280 stop there too).
__global__ void __launch_bounds__(256) k_reach(DevBuffers buf, DevParams prm) {
  const int b = blockIdx.y;
  const ScanOut& out = buf.out[b];
  ScanTab& tab = buf.tab[b];
  const int R = out.n_rings;
  const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = lane_id();
  if (w >= 2 * kDegBins || R <= 0) return;
  const int dir = w / kDegBins, i = w % kDegBins;
  if (dir == 0 ? i > prm.fwd_last : i < prm.bwd_first) return;          // outside the loop range: never accepted anyway
  const size_t nb = (size_t)prm.channels * kDegBins;
  CurbView cv{buf.cmin + (size_t)b * nb, buf.cmax + (size_t)b * nb, buf.ne + (size_t)b * prm.channels * (kDegBins + 1)};
  int reach = R;
  for (int k0 = 0; k0 < R; k0 += 32) {
    const int k = k0 + lane;
    const bool blocked = k < R && window_blocked(prm, cv, tab.A[k], dir, i, k);
    const unsigned bal = __ballot_sync(0xffffffffu, blocked);
    if (bal) { reach = k0 + __ffs(bal) - 1; break; }
  }
  if (lane == 0) tab.reach[dir][i] = reach;
}

// k_tab2: one warp per (ring, direction) builds a row of a threshold table with a warp max/min scan over the 361
// window starts (same result as the sequential build_T_row of urf_logic.cuh). Degree-major layout in memory: entry (j, k)
// at (j * channels + k) — a warp of k_label reads one or a few contiguous runs whether the sensor emits column-major (32
// rings at one azimuth) or ring-major (one ring, a few degrees). A CTA builds the rows of kTab2Rings consecutive rings in
// shared memory and writes them out transposed, kTab2Rings consecutive floats per degree.
constexpr int kTab2Rings = 16;
__global__ void __launch_bounds__(kTab2Rings * 64) k_tab2(DevBuffers buf, DevParams prm) {
  const int b = blockIdx.y;
  const ScanOut& out = buf.out[b];
  const ScanTab& tab = buf.tab[b];
  __shared__ float s_T[2][kDegBins][kTab2Rings + 1];     // +1: the row writes of a warp (stride kTab2Rings + 1) avoid bank conflicts
  const int w = threadIdx.x >> 5, lane = lane_id();
  const int kl = w >> 1, dir = w & 1;
  const int k0 = blockIdx.x * kTab2Rings, k = k0 + kl;
  const int R = out.n_rings;
  if (k0 >= R) return;
  constexpr int NCH = (kDegBins + 31) / 32;
  if (k < R) {
    const double A = tab.A[k];
    if (dir == 0) {
      int carry = -1;
      for (int c = 0; c < NCH; c++) {
        const int j = c * 32 + lane;
        int m = (j < kDegBins && accepted_fwd(prm, tab.reach[0], tab.q, k, j)) ? j : -1;
        for (int d = 1; d < 32; d <<= 1) { const int v = __shfl_up_sync(0xffffffffu, m, d); if (lane >= d) m = max(m, v); }
        m = max(m, carry);
        if (j < kDegBins) s_T[0][j][kl] = T_fwd_value(prm, k, m, A);
        carry = __shfl_sync(0xffffffffu, m, 31);
      }
    } else {
      int carry = 361;
      for (int c = NCH - 1; c >= 0; c--) {
        const int j = c * 32 + lane;
        int m = (j < kDegBins && accepted_bwd(prm, tab.reach[1], tab.q, k, j)) ? j : 361;
        for (int d = 1; d < 32; d <<= 1) { const int v = __shfl_down_sync(0xffffffffu, m, d); if (lane + d < 32) m = min(m, v); }
        m = min(m, carry);
        if (j < kDegBins) s_T[1][j][kl] = T_bwd_value(prm, k, m, A);
        carry = __shfl_sync(0xffffffffu, m, 0);
      }
    }
  }
  __syncthreads();
  const size_t ch = prm.channels;
  const size_t o = (size_t)b * ch * kTStride + k0;
  const int nk = min(kTab2Rings, R - k0);
  for (int t = threadIdx.x; t < 2 * kDegBins * kTab2Rings; t += blockDim.x) {
    const int kk = t % kTab2Rings, j = (t / kTab2Rings) % kDegBins, d = t / (kTab2Rings * kDegBins);
    if (kk < nk) (d == 0 ? buf.Tf : buf.Tb)[o + (size_t)j * ch + kk] = s_T[d][j][kk];
  }
}

// k_label: final label per input point, in input order (coalesced): -1 outside the ROI cloud, 2 where a detector marked
// the point, 1 where a blindSpots window covers it (two threshold look-ups, covered_from), else 0. Also the counts, per
// degree bin the first non-road point in the reference's scan order (ring, azimuth; equal azimuths in input order), and
// the road points for the marker search: every warp owns the 32 list slots at its own position (roadlist[warp * 32 ..],
// count in roadcnt[warp]) — no running counter, so no atomic with a return value and no barrier in this kernel: a warp's
// life is two memory round trips (its point's ring / azimuth / mark, then the two threshold entries and the bin's key).
__global__ void __launch_bounds__(256) k_label(DevBuffers buf, DevParams prm, int S) {
  const int b = blockIdx.y;
  ScanOut& out = buf.out[b];
  ScanTab& tab = buf.tab[b];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = buf.n[b];
  if ((i & ~31) >= n) return;                           // whole warp past the end of the scan
  const unsigned gb = scan_base(b, S), g = gb + (unsigned)i;
  int lab = -2, k = -2, bin = -1;                       // -2: past the end of the scan
  float a = 0.f, d = 0.f;
  unsigned long long key = ~0ull, cb = 0ull;            // first-non-road key of this point (~0 = none), current key of its bin
  if (i < n) {
    k = buf.ringid[g];
    lab = k == -2 ? URF_LABEL_OUTSIDE : URF_LABEL_NONE;
    if (k >= 0) {
      a = buf.az[g];
      d = buf.d2[g];
      const int m = buf.mark[g];
      // everything the decision needs is loaded up front (independent loads, one round trip): the two threshold entries
      // (degree-major table, see k_tab2) and, further down, the bin's current first-non-road key
      const unsigned o = (unsigned)b * (unsigned)prm.channels * kTStride + (unsigned)k;
      const bool valid = a >= 0.0f;
      int j = 0, jc = 0;
      if (valid) T_indices(a, &j, &jc);
      const float tf = buf.Tf[o + (unsigned)j * prm.channels], tb = buf.Tb[o + (unsigned)jc * prm.channels];
      if (valid) cb = __ldcg(&tab.cutbest[j]);          // from L2: L1 would keep serving the value of the first look
      lab = m == 2 ? 2 : (valid && covered_from(a, tf, tb)) ? 1 : 0;   // covered_T of urf_logic.cuh with the loads hoisted
      if (valid) bin = j;                               // == deg_bin(a)
      if (valid && lab != 1) key = best_key(k, fbits(a), i);          // lidar_segmentation.cpp:318: non-road point in bin [i, i+1)
    }
    buf.label[g] = lab;
    if (buf.label8) buf.label8[g] = (signed char)lab;
    if (prm.want_order && i >= out.n_order) buf.order[g] = -1;   // defined tail of the emission order (k_sort_rings writes [0, n_order))
  }
  // first non-road point per bin: atomicMin of the keys. A column-major scan puts the 32 rings of one azimuth — one bin —
  // into a warp, a ring-major one a few neighbouring bins: when all keys of the warp belong to one bin only their minimum
  // goes out (one atomic per warp instead of one per point).
  const bool has_key = key != ~0ull;
  const unsigned hk = __ballot_sync(0xffffffffu, has_key);
  if (hk) {
    const int bin0 = __shfl_sync(0xffffffffu, bin, __ffs(hk) - 1);
    if (__all_sync(0xffffffffu, !has_key || bin == bin0)) {
      const unsigned hi = (unsigned)(key >> 32), mh = __reduce_min_sync(0xffffffffu, hi);
      const unsigned ml = __reduce_min_sync(0xffffffffu, hi == mh ? (unsigned)key : 0xffffffffu);
      const unsigned long long cb0 = __shfl_sync(0xffffffffu, cb, __ffs(hk) - 1);
      if (lane_id() == 0) {
        const unsigned long long mk = ((unsigned long long)mh << 32) | ml;
        if (cb0 > mk) atomicMin(&tab.cutbest[bin0], mk);
      }
    } else if (has_key && cb > key) atomicMin(&tab.cutbest[bin], key);
  }
  const unsigned br = __ballot_sync(0xffffffffu, lab == 1), bc = __ballot_sync(0xffffffffu, lab == 2);
  if (lane_id() == 0) {
    buf.roadcnt[(size_t)b * ((S + 31) >> 5) + (unsigned)(i >> 5)] = (unsigned char)__popc(br);
    if (br) atomicAdd(&out.n_road, __popc(br));         // results unused: fire-and-forget
    if (bc) atomicAdd(&out.n_curb, __popc(bc));
  }
  if (lab == 1)
    buf.roadlist[gb + (unsigned)(i & ~31) + (unsigned)__popc(br & ((1u << lane_id()) - 1u))] =
        make_uint4((unsigned)bin | ((unsigned)k << 16), fbits(a), fbits(d), (unsigned)i);
}

// k_markers1: marker candidate vertices, lidar_segmentation.cpp:305-351, over the road points k_label listed (32 slots per
// warp of input points, count in roadcnt) — ONE CTA of 1024 threads per scan, everything in its own shared memory:
//   pass 1  farthest candidate road point per bin (candidates: road points scanned before the bin's first non-road point)
//   pass 2  first candidate in scan order that reaches that distance (`d > maxDistanceRoad` is strict, :329)
//   then    the per-bin winners are compacted in bin order into markerPointsArray (:343-350)
// In a pass a warp takes 32 list segments at a time, scans their counts and spreads the entries evenly over its lanes
// (entry e of the 32 segments belongs to the segment whose exclusive count prefix is the last one <= e), four entries in
// flight per lane. (Measured and dropped: a cluster of eight CTAs per scan merging through distributed shared memory,
// 0.077 ms against 0.052 ms, its cluster barriers dominating the stall samples.)
constexpr int kMark1Threads = 1024;
template <int PASS>
__device__ __forceinline__ void markers_pass(const uint4* __restrict__ list, const unsigned char* __restrict__ cnt, int nseg,
                                             const unsigned long long* s_cut, unsigned* s_dmax, unsigned long long* s_best) {
  const int lane = lane_id(), nwarps = (blockDim.x >> 5) * gridDim.x;       // warps of all CTAs that share this scan
  const int warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int cpre[4];                                          // counts of the warp's next four sweeps, loaded together
  for (int seg0 = warp * 32, sw = 0; seg0 < nseg; seg0 += nwarps * 32, sw++) {
    if ((sw & 3) == 0) {
#pragma unroll
      for (int u = 0; u < 4; u++) { const int sg = seg0 + u * nwarps * 32 + lane; cpre[u] = sg < nseg ? cnt[sg] : 0; }
    }
    const int c = (sw & 3) == 0 ? cpre[0] : (sw & 3) == 1 ? cpre[1] : (sw & 3) == 2 ? cpre[2] : cpre[3];
    int inc = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
    const int excl = inc - c, total = __shfl_sync(0xffffffffu, inc, 31);
    for (int e0 = 0; e0 < total; e0 += 128) {
      uint4 ent[4];
      bool ok[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int e = e0 + u * 32 + lane;
        int lo = 0;                                      // last segment whose exclusive prefix is <= e (skips empty segments)
#pragma unroll
        for (int step = 16; step > 0; step >>= 1) {
          const int ex = __shfl_sync(0xffffffffu, excl, lo + step < 32 ? lo + step : 31);
          if (lo + step < 32 && ex <= e) lo += step;
        }
        const int r = e - __shfl_sync(0xffffffffu, excl, lo);
        ok[u] = e < total;
        ent[u] = ok[u] ? list[(seg0 + lo) * 32 + r] : make_uint4(0u, 0u, 0u, 0u);
      }
#pragma unroll
      for (int u = 0; u < 4; u++) {
        if (!ok[u]) continue;
        const uint4 q = ent[u];
        const int bin = q.x & 0xffff, k = q.x >> 16;
        if (PASS == 1) {
          if (marker_candidate(s_cut[bin], k, q.y, (int)q.w) && s_dmax[bin] < q.z) atomicMax(&s_dmax[bin], q.z);
        } else if (q.z != 0u && q.z == s_dmax[bin] && marker_candidate(s_cut[bin], k, q.y, (int)q.w)) {
          const unsigned long long key = best_key(k, q.y, (int)q.w);
          if (s_best[bin] > key) atomicMin(&s_best[bin], key);
        }
      }
    }
  }
}
__global__ void __launch_bounds__(kMark1Threads) k_markers1(DevBuffers buf, int S) {
  const int b = blockIdx.y;                            // grid (1, B)
  ScanOut& out = buf.out[b];
  const ScanTab& tab = buf.tab[b];
  __shared__ unsigned long long s_cut[kDegBins], s_best[kDegBins];
  __shared__ unsigned s_dmax[kDegBins];
  __shared__ int s_wsum[kMark1Threads / 32];
  const int tid = threadIdx.x;
  for (int t = tid; t < kDegBins; t += kMark1Threads) { s_cut[t] = tab.cutbest[t]; s_dmax[t] = 0u; s_best[t] = ~0ull; }
  __syncthreads();
  const int n = buf.n[b];
  const int nseg = (n + 31) >> 5;
  const unsigned char* cnt = buf.roadcnt + (size_t)b * ((S + 31) >> 5);
  const uint4* list = buf.roadlist + scan_base(b, S);
  markers_pass<1>(list, cnt, nseg, s_cut, s_dmax, s_best);
  __syncthreads();
  markers_pass<2>(list, cnt, nseg, s_cut, s_dmax, s_best);
  __syncthreads();
  const int i = tid;                                   // kMark1Threads >= kDegBins: one bin per thread
  const bool has = i < kDegBins && s_best[i] != ~0ull;
  const unsigned bal = __ballot_sync(0xffffffffu, has);
  const int warp = i >> 5, lane = lane_id();
  if (lane == 0) s_wsum[warp] = __popc(bal);
  __syncthreads();
  int off = 0, total = 0;
  for (int w = 0; w < kMark1Threads / 32; w++) { if (w < warp) off += s_wsum[w]; total += s_wsum[w]; }
  if (has) {
    const int slot = off + __popc(bal & ((1u << lane) - 1u));
    const int p = (int)(s_best[i] & 0xffffffull);      // input index of the winner
    const float4 q = buf.in[(size_t)b * S + p];
    out.vert[slot][0] = q.x; out.vert[slot][1] = q.y; out.vert[slot][2] = q.z;
    out.vert[slot][3] = s_cut[i] != ~0ull ? 1.0f : 0.0f;                // redPoints, :320,348
  }
  if (i == 0) out.n_vert = total;
  if (i >= total && i < URF_MAX_VERTS) { out.vert[i][0] = 0.f; out.vert[i][1] = 0.f; out.vert[i][2] = 0.f; out.vert[i][3] = 0.f; }   // defined tail
}

// The same search for LARGE scans (hundreds of thousands of road points want more than one CTA): a grid of CTAs per scan,
// every CTA aggregates its share per degree bin in shared memory and merges into the scan's global arrays with atomics;
// pass 1, pass 2 and the vertex compaction are three launches.
constexpr int kMarkGridThreads = 256;
template <int PASS>
__global__ void __launch_bounds__(kMarkGridThreads) k_markers_grid(DevBuffers buf, int S) {
  const int b = blockIdx.y;
  ScanTab& tab = buf.tab[b];
  __shared__ unsigned long long s_cut[kDegBins], s_best[kDegBins];
  __shared__ unsigned s_dmax[kDegBins];
  const int tid = threadIdx.x;
  for (int t = tid; t < kDegBins; t += kMarkGridThreads) {
    s_cut[t] = tab.cutbest[t]; s_best[t] = ~0ull;
    s_dmax[t] = PASS == 1 ? 0u : tab.dmax[t];          // pass 2 compares with the merged maxima of pass 1
  }
  __syncthreads();
  const int n = buf.n[b];
  const int nseg = (n + 31) >> 5;
  const unsigned char* cnt = buf.roadcnt + (size_t)b * ((S + 31) >> 5);
  const uint4* list = buf.roadlist + scan_base(b, S);
  markers_pass<PASS>(list, cnt, nseg, s_cut, s_dmax, s_best);
  __syncthreads();
  for (int t = tid; t < kDegBins; t += kMarkGridThreads) {
    if (PASS == 1) { const unsigned v = s_dmax[t]; if (v) atomicMax(&tab.dmax[t], v); }
    else { const unsigned long long v = s_best[t]; if (v != ~0ull) atomicMin(&tab.best[t], v); }
  }
}
// k_verts: compact the per-bin winners (tab.best) in bin order into markerPointsArray (lidar_segmentation.cpp:343-350)
__global__ void __launch_bounds__(384) k_verts(DevBuffers buf, int S) {
  const int b = blockIdx.x;
  ScanOut& out = buf.out[b];
  const ScanTab& tab = buf.tab[b];
  __shared__ int s_wsum[12];
  const int i = threadIdx.x;
  const bool has = i < kDegBins && tab.best[i] != ~0ull;
  const unsigned bal = __ballot_sync(0xffffffffu, has);
  const int warp = i >> 5, lane = lane_id();
  if (lane == 0) s_wsum[warp] = __popc(bal);
  __syncthreads();
  int off = 0, total = 0;
  for (int w = 0; w < 12; w++) { if (w < warp) off += s_wsum[w]; total += s_wsum[w]; }
  if (has) {
    const int slot = off + __popc(bal & ((1u << lane) - 1u));
    const int p = (int)(tab.best[i] & 0xffffffull);    // input index of the winner
    const float4 q = buf.in[(size_t)b * S + p];
    out.vert[slot][0] = q.x; out.vert[slot][1] = q.y; out.vert[slot][2] = q.z;
    out.vert[slot][3] = tab.cutbest[i] != ~0ull ? 1.0f : 0.0f;          // redPoints, :320,348
  }
  if (i == 0) out.n_vert = total;
  if (i >= total && i < URF_MAX_VERTS) { out.vert[i][0] = 0.f; out.vert[i][1] = 0.f; out.vert[i][2] = 0.f; out.vert[i][3] = 0.f; }   // defined tail
}

// ---------------------------------------------------------------------------------------------------------------------
// k_sort_rings (only when the emission order is requested): per-ring sort by azimuth, lidar_segmentation.cpp:70-93,289-291.
// Tie policy: (azimuth, input order) — the reference's Lomuto quicksort is unstable; ties raise F_TIE_AZIMUTH.
// One CTA per ring. Rings of up to kRingFast points take a counting sort in shared memory: azimuths are spread over
// kRingBins equal-width bins between the ring's smallest and largest azimuth (a monotone map, so bin order = azimuth
// order), a histogram + exclusive scan places every point in its bin, and the few points that share a bin (LiDAR rings
// are close to uniform in azimuth) are ordered by one thread with an insertion sort on (azimuth bits, position). A ring
// with a crowded bin (more than kBinCap points) or more than kRingFast points falls back to the CTA-wide bitonic sort on
// 64-bit (azimuth bits, position) keys. Both paths produce the same total order.
constexpr int kRingSmemKeys = 6144;                     // 48 KB of dynamic shared memory: four CTAs per SM
constexpr int kRingFast = 4096, kRingBins = 4096, kBinCap = 48;
constexpr int kSortThreads = 512;
__global__ void __launch_bounds__(kSortThreads) k_sort_rings(DevBuffers buf, int S) {
  extern __shared__ unsigned long long s_rkeys[];
  const int b = blockIdx.y, k = blockIdx.x;
  ScanOut& out = buf.out[b];
  if (k >= out.n_rings) return;
  const int base = out.ring_start[k], n = out.ring_start[k + 1] - base;
  if (n <= 0) return;
  const size_t gb = (size_t)b * S, g0 = gb + base;
  const int tid = threadIdx.x;
  if (n <= kRingFast) {
    unsigned* s_az = reinterpret_cast<unsigned*>(s_rkeys);            // [kRingFast] azimuth bits by ring position
    unsigned* s_cnt = s_az + kRingFast;                               // [kRingBins] bin counts, then exclusive starts
    unsigned short* s_rank = reinterpret_cast<unsigned short*>(s_cnt + kRingBins);   // [kRingFast] arrival rank inside the bin
    unsigned short* s_slot = s_rank + kRingFast;                      // [kRingFast] ring position by sorted position
    __shared__ unsigned s_lo, s_hi, s_over, s_wsum[kSortThreads / 32];
    if (tid == 0) { s_lo = 0xffffffffu; s_hi = 0u; s_over = 0u; }
    for (int t = tid; t < kRingBins; t += kSortThreads) s_cnt[t] = 0u;
    __syncthreads();
    unsigned lo = 0xffffffffu, hi = 0u;
    for (int t0 = tid; t0 < n; t0 += 4 * kSortThreads) {             // four coalesced loads in flight per thread
      unsigned av[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int t = t0 + u * kSortThreads;
        av[u] = t < n ? buf.baz[g0 + t].x : 0u;                      // (azimuth, input index) in bucket order, written by k_scatter
      }
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int t = t0 + u * kSortThreads;
        if (t < n) {
          s_az[t] = av[u];
          if (av[u] <= 0x7f800000u) { lo = min(lo, av[u]); hi = max(hi, av[u]); }   // azimuths are >= +0: their bits order them; NaN stays out
        }
      }
    }
    lo = __reduce_min_sync(0xffffffffu, lo); hi = __reduce_max_sync(0xffffffffu, hi);
    if (lane_id() == 0) { atomicMin(&s_lo, lo); atomicMax(&s_hi, hi); }
    __syncthreads();
    const float flo = bitsf(s_lo), fhi = bitsf(s_hi);
    const float scale = fhi > flo ? __fdiv_rn((float)(kRingBins - 2), __fsub_rn(fhi, flo)) : 0.0f;
    auto bin_of = [&](unsigned a) -> int {                           // monotone in a; NaN azimuths go to the last bin
      if (a > 0x7f800000u) return kRingBins - 1;
      const int v = __float2int_rz(__fmul_rn(__fsub_rn(bitsf(a), flo), scale));
      return v < 0 ? 0 : (v > kRingBins - 2 ? kRingBins - 2 : v);
    };
    for (int t = tid; t < n; t += kSortThreads) s_rank[t] = (unsigned short)atomicAdd(&s_cnt[bin_of(s_az[t])], 1u);
    __syncthreads();
    {   // exclusive scan over the bins: consecutive bins per thread, warp scan, warp totals
      constexpr int PER = kRingBins / kSortThreads;
      unsigned v[PER], sum = 0, mx = 0;
#pragma unroll
      for (int j = 0; j < PER; j++) { v[j] = s_cnt[tid * PER + j]; sum += v[j]; mx = max(mx, v[j]); }
      if (mx > (unsigned)kBinCap) s_over = 1u;
      unsigned inc = sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const unsigned y = __shfl_up_sync(0xffffffffu, inc, o); if (lane_id() >= o) inc += y; }
      if (lane_id() == 31) s_wsum[tid >> 5] = inc;
      __syncthreads();
      unsigned run = inc - sum;
      for (int w = 0; w < (tid >> 5); w++) run += s_wsum[w];
#pragma unroll
      for (int j = 0; j < PER; j++) { s_cnt[tid * PER + j] = run; run += v[j]; }
    }
    __syncthreads();
    if (!s_over) {
      for (int t = tid; t < n; t += kSortThreads) s_slot[s_cnt[bin_of(s_az[t])] + s_rank[t]] = (unsigned short)t;
      __syncthreads();
      constexpr int PER = kRingBins / kSortThreads;
      for (int j = 0; j < PER; j++) {                                  // order the points that share a bin
        const int bin = tid * PER + j;
        const int s0 = (int)s_cnt[bin], s1 = bin + 1 < kRingBins ? (int)s_cnt[bin + 1] : n;
        for (int e = s0 + 1; e < s1; e++) {
          const unsigned short cur = s_slot[e];
          const unsigned ca = s_az[cur];
          int f = e - 1;
          while (f >= s0) {
            const unsigned short o = s_slot[f];
            const unsigned oa = s_az[o];
            if (oa < ca || (oa == ca && o < cur)) break;
            s_slot[f + 1] = o; f--;
          }
          s_slot[f + 1] = cur;
        }
      }
      __syncthreads();
      bool tie = false;
      for (int p = tid; p < n; p += kSortThreads) {
        const unsigned short slot = s_slot[p];
        buf.order[g0 + p] = (int)buf.baz[g0 + slot].y;               // the ring's pairs are in L2 from the first pass
        if (p > 0 && s_az[s_slot[p - 1]] == s_az[slot]) tie = true;
      }
      if (tie) atomicOr(&out.flags, F_TIE_AZIMUTH);
      return;
    }
    __syncthreads();                                                   // the fallback reuses the shared memory
  }
  const int npad = next_pow2(n < 2 ? 2 : n);
  unsigned long long* keys = npad <= kRingSmemKeys ? s_rkeys : buf.sortbuf + 2 * g0;
  for (int t = tid; t < npad; t += blockDim.x)
    keys[t] = t < n ? (((unsigned long long)buf.baz[g0 + t].x << 32) | (unsigned)t) : ~0ull;
  __syncthreads();
  cta_bitonic(keys, npad);
  bool tie = false;
  for (int t = tid; t < n; t += blockDim.x) {
    const unsigned long long key = keys[t];
    buf.order[g0 + t] = (int)buf.baz[g0 + (unsigned)key].y;
    if (t > 0 && (unsigned)(keys[t - 1] >> 32) == (unsigned)(key >> 32)) tie = true;
  }
  if (tie) atomicOr(&out.flags, F_TIE_AZIMUTH);
}

// k_unpack_cloud2: PointCloud2 record -> (x, y, z, intensity) float4 (SURVEY.md §8 f1). Byte-wise loads when a field is
// not 4-byte aligned (Velodyne's 22-byte records). off_i < 0: no intensity field, 0 is stored.
__device__ __forceinline__ float load_f32_unaligned(const unsigned char* p) {
  if ((reinterpret_cast<size_t>(p) & 3) == 0) return *reinterpret_cast<const float*>(p);
  const unsigned v = (unsigned)p[0] | ((unsigned)p[1] << 8) | ((unsigned)p[2] << 16) | ((unsigned)p[3] << 24);
  return __uint_as_float(v);
}
__global__ void __launch_bounds__(256) k_unpack_cloud2(const unsigned char* __restrict__ raw, float4* __restrict__ dst, int n,
                                                        int point_step, int off_x, int off_y, int off_z, int off_i) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned char* rec = raw + (size_t)i * point_step;
  dst[i] = make_float4(load_f32_unaligned(rec + off_x), load_f32_unaligned(rec + off_y), load_f32_unaligned(rec + off_z),
                       off_i >= 0 ? load_f32_unaligned(rec + off_i) : 0.f);
}
// the same for a batch: scan b = blockIdx.y, its records at raw + b * S * point_step, its points at dst + b * S
__global__ void __launch_bounds__(256) k_unpack_cloud2_batch(const unsigned char* __restrict__ raw, float4* __restrict__ dst,
                                                              const int* __restrict__ n, int S, int point_step, int off_x, int off_y,
                                                              int off_z, int off_i) {
  const int b = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n[b]) return;
  const unsigned char* rec = raw + ((size_t)b * S + i) * point_step;
  dst[(size_t)b * S + i] = make_float4(load_f32_unaligned(rec + off_x), load_f32_unaligned(rec + off_y), load_f32_unaligned(rec + off_z),
                                       off_i >= 0 ? load_f32_unaligned(rec + off_i) : 0.f);
}

// ---------------------------------------------------------------------------------------------------------------------
// Output clouds packed on the device (SURVEY.md §8 f1, scan 0 of the buffers): what lidar_segmentation.cpp:354-367 and
// :605-608 push into cloud_filtered_Road / _High / _ProbablyRoad and what :120 leaves in cloud_filtered_Box, as 32-byte
// pcl::PointXYZI records (x, y, z, 1.0f | intensity, 0, 0, 0) in the reference's emission order:
//   road = points of `order` (ring-major, ascending azimuth) with label 1, curb = label 2 (stored behind road in the same
//   buffer), roi = label >= 0 in input order, road_probably = ring 10 of `order`.
// Three kernels: per-tile counts -> exclusive scan over tiles -> stable per-tile compaction.
constexpr int kPackTile = 1024;
__device__ __forceinline__ void pack_flags(const DevBuffers& buf, const ScanOut& out, int e, bool* road, bool* curb, bool* roi, int* idx) {
  *road = *curb = *roi = false; *idx = 0;
  if (out.n_roi < 30) return;                                            // nothing is published, lidar_segmentation.cpp:124-126
  if (e < out.n_order) { *idx = buf.order[e]; const int lab = buf.label[*idx]; *road = lab == 1; *curb = lab == 2; }
  if (e < out.n_in) *roi = buf.label[e] >= 0;
}
// exclusive rank of `flag` among the CTA's 256 threads (thread order) and the CTA total; all threads must call
__device__ __forceinline__ int cta_rank(bool flag, int* s_w /* [8] */, int* total) {
  const unsigned bal = __ballot_sync(0xffffffffu, flag);
  const int w = threadIdx.x >> 5;
  __syncthreads();                                                       // s_w free again
  if (lane_id() == 0) s_w[w] = __popc(bal);
  __syncthreads();
  int before = 0, all = 0;
#pragma unroll
  for (int j = 0; j < 8; j++) { const int c = s_w[j]; all += c; if (j < w) before += c; }
  *total = all;
  return before + __popc(bal & ((1u << lane_id()) - 1u));
}
__global__ void __launch_bounds__(256) k_pack_count(DevBuffers buf, int* __restrict__ cnt, int tiles) {
  __shared__ int s_c[3];
  const ScanOut& out = buf.out[0];
  if (threadIdx.x < 3) s_c[threadIdx.x] = 0;
  __syncthreads();
  int c0 = 0, c1 = 0, c2 = 0;
  for (int j = 0; j < kPackTile / 256; j++) {
    bool road, curb, roi; int idx;
    pack_flags(buf, out, blockIdx.x * kPackTile + j * 256 + threadIdx.x, &road, &curb, &roi, &idx);
    c0 += road; c1 += curb; c2 += roi;
  }
  c0 = __reduce_add_sync(0xffffffffu, c0); c1 = __reduce_add_sync(0xffffffffu, c1); c2 = __reduce_add_sync(0xffffffffu, c2);
  if (lane_id() == 0) { atomicAdd(&s_c[0], c0); atomicAdd(&s_c[1], c1); atomicAdd(&s_c[2], c2); }
  __syncthreads();
  if (threadIdx.x < 3) cnt[threadIdx.x * tiles + blockIdx.x] = s_c[threadIdx.x];
}
// one CTA: exclusive scan of the three per-tile count rows in place; tot[0..3] = road, curb, roi, road_probably counts
__global__ void __launch_bounds__(1024) k_pack_scan(DevBuffers buf, int* __restrict__ cnt, int tiles, int* __restrict__ tot) {
  __shared__ int s_w[32];
  __shared__ int s_carry;
  for (int row = 0; row < 3; row++) {
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int t0 = 0; t0 < tiles; t0 += 1024) {
      const int t = t0 + threadIdx.x;
      const int v = t < tiles ? cnt[row * tiles + t] : 0;
      int x = v;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, d); if (lane_id() >= d) x += y; }
      if (lane_id() == 31) s_w[threadIdx.x >> 5] = x;
      __syncthreads();
      if (threadIdx.x < 32) {
        int wv = s_w[threadIdx.x];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(0xffffffffu, wv, d); if (lane_id() >= d) wv += y; }
        s_w[threadIdx.x] = wv;
      }
      __syncthreads();
      const int carry = s_carry, wbase = (threadIdx.x >> 5) ? s_w[(threadIdx.x >> 5) - 1] : 0;
      if (t < tiles) cnt[row * tiles + t] = carry + wbase + x - v;
      __syncthreads();
      if (threadIdx.x == 0) s_carry = carry + s_w[31];
      __syncthreads();
    }
    if (threadIdx.x == 0) tot[row] = s_carry;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const ScanOut& out = buf.out[0];
    tot[3] = out.n_roi < 30 ? 0 : out.ring_start[11] - out.ring_start[10];     // lidar_segmentation.cpp:605-608
  }
}
__device__ __forceinline__ void pack_record(float4* __restrict__ dst, int pos, const float4 p) {
  dst[2 * (size_t)pos] = make_float4(p.x, p.y, p.z, 1.0f);               // PCL_ADD_POINT4D: data[3] = 1.0f
  dst[2 * (size_t)pos + 1] = make_float4(p.w, 0.f, 0.f, 0.f);            // intensity + padding
}
__global__ void __launch_bounds__(256) k_pack_write(DevBuffers buf, const int* __restrict__ cnt, int tiles, const int* __restrict__ tot,
                                                     float4* __restrict__ road_curb, float4* __restrict__ roi_dst, float4* __restrict__ prob) {
  __shared__ int s_w[8];
  const ScanOut& out = buf.out[0];
  int road_pos = cnt[blockIdx.x], curb_pos = tot[0] + cnt[tiles + blockIdx.x], roi_pos = cnt[2 * tiles + blockIdx.x];
  const int rs10 = out.ring_start[10], rs11 = out.n_roi < 30 ? rs10 : out.ring_start[11];
  for (int j = 0; j < kPackTile / 256; j++) {
    const int e = blockIdx.x * kPackTile + j * 256 + threadIdx.x;
    bool road, curb, roi; int idx;
    pack_flags(buf, out, e, &road, &curb, &roi, &idx);
    int total;
    const int r0 = cta_rank(road, s_w, &total);
    if (road) pack_record(road_curb, road_pos + r0, buf.in[idx]);
    road_pos += total;
    const int r1 = cta_rank(curb, s_w, &total);
    if (curb) pack_record(road_curb, curb_pos + r1, buf.in[idx]);
    curb_pos += total;
    const int r2 = cta_rank(roi, s_w, &total);
    if (roi) pack_record(roi_dst, roi_pos + r2, buf.in[e]);
    roi_pos += total;
    if (e >= rs10 && e < rs11) pack_record(prob, e - rs10, buf.in[idx]);
  }
}

// Device-side evaluation of the emulated libm (test hook: urf_test_math).
__global__ void k_test_math(const float* a, const float* bb, float* o, int n, int which) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float r;
  switch (which) {
    case 0: r = urfm::asinf_glibc(a[i]); break;
    case 1: r = urfm::acosf_glibc(a[i]); break;
    case 2: r = urfm::atan2f_glibc(a[i], bb[i]); break;
    default: r = urfm::atanf_glibc(a[i]); break;
  }
  o[i] = r;
}

}  // namespace urf
