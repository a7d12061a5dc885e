// urf_device.cuh — device-side data layout of liburf_b200 (see DESIGN.md "Data layout in HBM").
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/urf.h"

namespace urf {

constexpr int kChunk = 512;           // input points per warp chunk in the stable partition kernels
constexpr int kWarpsPerBlock = 8;     // chunks per CTA in the partition kernels
constexpr int kRingKeys = URF_MAX_CHANNELS;                 // 256 ring keys
constexpr int kSectKeys = URF_STAR_SECTORS;                 // 360 sector keys
constexpr int kElevBins = 4096;       // fine elevation bins used to speculate the greedy ring registration
constexpr int kMaxCand = 1024;        // max speculation candidates handled by the fast registration path
constexpr int kDegBins = 361;         // integer-degree bins 0..360 (marker search, lidar_segmentation.cpp:305)
constexpr int kStLevels = 9;          // sparse-table levels over 361 window starts (CPU model cross-check only)

// per-scan flag bits: the low 4 bits are the public urf_result.flags, the rest is internal
enum : int {
  F_EXACT_REG = 1,       // exact (sequential-semantics) ring registration was used
  F_TIE_SECTOR = 2,      // a star sector holds two points with identical planar radius AMONG THE POINTS THAT WERE SORTED (the
                         // near-first sort leaves the far part of a sector unsorted: ties there are neither seen nor relevant)
  F_TIE_AZIMUTH = 4,     // a ring holds two points with identical azimuth (only detected when `order` is produced)
  F_NAN_AZIMUTH = 8,     // a ROI point has x == y == 0: its azimuth is NaN (DESIGN.md deviation 3: the reference's window scans
                         // stop at such a point and its quicksort places it unpredictably; here it belongs to no window or bin)
  F_ZERO_ALPHA = 16,     // an elevation angle of exactly 0 exists (reference's `angle[j]==0` sentinel quirk) -> exact path
  F_SPEC_VIOLATION = 32, // speculative registration failed verification -> exact path + re-assignment
  F_PUBLIC_MASK = 15
};

// Narrowed parameters (src/main.cpp:5-32 narrows every double to float) plus host-derived loop bounds.
struct DevParams {
  int x_zero, z_zero, star, blind, xDirection;
  float interval, curbHeight;
  int curbPoints;
  float beamZone, angleFilter1, angleFilter2, slope_param;
  float min_X, max_X, min_Y, max_Y, min_Z, max_Z;
  float kdev, kdist;
  int starbeam, dmin, channels;
  float Kfi;
  // blind_spots.cpp:68 `for (i = 0; i <= 360 - beamZone; i++)` and :177 `for (i = 360; i >= 0 + beamZone; --i)`
  int fwd_last;      // largest i >= 0 with (float)i <= 360.0f - beamZone, or -1
  int fwd_special;   // the i with (float)i == 360.0f - beamZone (:136), or -1
  int bwd_first;     // smallest i <= 360 with (float)i >= beamZone, or 361
  int bwd_special;   // the i with (float)i == beamZone (:245), or -1
  int force_exact;   // test hook: always use the exact registration path
  int want_order;    // produce emission order (per-ring azimuth sort)
  int star_prefix;   // near-first star sort on (default); 0 = always sort whole sectors (test hook)
};

// Near-first star sort: rank (0..31) of the pivot among 32 evenly spaced radius samples of a sector, here the 18th
// smallest (tighter and looser pivots measured slower or equal, DESIGN.md §6). The eight-warp sort takes rank
// 8 * kStarPivot + 7 of 256 samples.
constexpr int kStarPivot = 17;

// Small per-scan outputs copied back to the host after every call.
struct ScanOut {
  int n_in, n_roi, n_rings, n_order, n_road, n_curb, n_vert, flags;
  int ring_start[kRingKeys + 1];
  float vert[URF_MAX_VERTS][4];
};

// Per-scan working tables that stay on the device.
struct ScanTab {
  float angle[kRingKeys];          // sorted registered elevation angles (lidar_segmentation.cpp:205)
  int regidx[kRingKeys];           // input index that registered angle[j]
  int regorder[kRingKeys];         // registration input indices in registration (= ascending) order
  unsigned long long maxs[kRingKeys];   // bits of the ring's largest (double)x*x + y*y (k_ring_detect); see planar_sum_bits
  unsigned maxdist[kRingKeys];     // float bits of maxDistance[j] (:271-274) = (float)sqrt(maxs[j]), taken in k_tab1
  double A[kRingKeys];             // arcDistance / ((maxDistance[k] * M_PI) / 180)  (blind_spots.cpp:142)
  int sect_start[kSectKeys + 1];
  int sect_cnt[kSectKeys];         // points per star sector (unstable partition: counted with atomics)
  int sect_cur[kSectKeys];         // scatter cursors
  int nbig, nslow;                 // work lists of the star sort: sectors for the CTA radix sort / the bitonic fallback
  unsigned short biglist[kSectKeys], slowlist[kSectKeys];
  float q[4];                      // q1..q4 (blind_spots.cpp:13-57)
  int reach[2][kDegBins];          // rings accepted by window start i, forward / backward (atomicMin over cells)
  unsigned long long cutbest[kDegBins];              // min (ring, azimuth bits, input index) over the bin's non-road points
  unsigned dmax[kDegBins];         // large scans (k_markers_grid): float bits of the farthest candidate road point
  unsigned long long best[kDegBins];                 // large scans: (ring, azimuth bits, input index) of the first candidate reaching dmax
  // near-first star sort (k_star_sort_warp): only the points below a sampled pivot radius are sorted at first
  int sorted_len[kSectKeys];       // length of the radius-sorted prefix of the sector in `ssorted` (== size when fully sorted)
  int nrefine, pad_;               // sectors whose edge search ran off the sorted prefix
  unsigned short refine[kSectKeys];
  float resume[kSectKeys][4];      // per refine entry: running mean, deviation, NaN count of the walk over the prefix, its length
};

// All device buffers of a context. P = max_batch * max_points; T = ceil(max_points / kChunk).
struct DevBuffers {
  float4* in;            // [P]   x, y, z, intensity (input order)
  float* alpha_v;        // [P]   elevation angle in degrees, -1 = outside ROI
  unsigned char* mark;   // [P]   detector mark per input point: 2 = curb (star-shaped, x-zero or z-zero), else 0
  short* ringid;         // [P]   ring index; -1 = in the ROI but no registered ring matches; -2 = not in the ROI cloud
  short* sect;           // [P]   star sector or -1
  int* label;            // [P]   output labels, input order
  signed char* label8;   // [P] or NULL: the same labels as one byte per point (callers that ask for int8 labels)
  float4* bpt;           // [P]   ring buckets (ring-major, input order inside a ring): x, y, z, input index bits
  float4* spt;           // [P]   sector buckets (unordered inside a sector): r, z, input index bits, -
  float4* ssorted;       // [P]   sector buckets sorted by r
  float* az;             // [P]   azimuth per input point (ROI points only)
  float* d2;             // [P]   planar range per input point (ROI points only)
  uint2* baz;            // [P]   (azimuth bits, input index) per bucket position (written by k_scatter only when the emission order is wanted)
  uint4* roadlist;       // [P]   road points, 32 slots per warp of input points: (bin | ring << 16, azimuth bits, range bits, input index)
  unsigned char* roadcnt; // [B][ceil(S / 32)] road points of each input warp (entries used in its 32 list slots)
  float* Tf;             // [B][channels][kTStride] forward threshold table (urf_logic.cuh build_T_row)
  float* Tb;             // [B][channels][kTStride] backward threshold table
  unsigned short* lut;   // [B][kElevBins + 1] ring-search start per fine elevation bin
  int* order;            // [P]   emission order (input indices), only when requested
  unsigned long long* sortbuf;   // [2P] scratch for segments too large for shared memory
  unsigned* hist;        // [B][T][kRingKeys] per-chunk ring histograms, turned into scatter offsets in place
  unsigned* firstidx;    // [B][kElevBins + 1] first input index per fine elevation bin
  unsigned* cmin;        // [B][channels][kDegBins] float bits: min curb azimuth per (ring, degree bin), +inf = empty
  unsigned* cmax;        // [B][channels][kDegBins] float bits: max curb azimuth per (ring, degree bin)
  unsigned short* ne;    // [B][channels][kDegBins + 1] prefix count of non-empty curb bins
  float* newY;           // [max_points] x-zero `newY` ramp (x_zero_method.cpp:24-27), depends on the index only
  int* n;                // [B] points per scan
  ScanOut* out;          // [B]
  ScanTab* tab;          // [B]
};

}  // namespace urf
