// urf_api.cu — host side of liburf_b200.so: context, parameter narrowing, pipeline launcher and the C-ABI of include/urf.h.
// There is no CPU fallback in this library: without a CUDA device every compute entry point returns an error.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "urf_kernels.cuh"
#include "urf_host.hpp"

using namespace urf;

struct urf_ctx {
  int device = 0;
  int max_points = 0;      // per scan, rounded up to kChunk
  int max_batch = 0;
  size_t P = 0;            // max_batch * max_points
  int Tmax = 0;
  cudaStream_t stream = nullptr;       // compute
  cudaStream_t s_in = nullptr, s_out = nullptr;   // H2D / D2H copy streams of the pipelined host-buffer path
  static constexpr int kGroups = 16;               // sub-batches of a device-resident call run on separate streams: scans are
  cudaStream_t s_grp[kGroups] = {};               // independent, so their (short, partly latency-bound) kernels overlap
  cudaEvent_t ev_fork = nullptr, ev_join[kGroups] = {};
  // inside one pipeline the star-shaped search (four kernels) and the ring detector (one kernel) are independent between
  // k_scatter and k_tab1: the ring detector runs on a side stream of the pipeline's stream (measured at C2 x 128:
  // 1.240 -> 1.233 ms on two streams, 1.282 -> 1.263 on one)
  cudaStream_t s_side[kGroups + 1] = {};
  cudaEvent_t ev_sfork[kGroups + 1] = {}, ev_sjoin[kGroups + 1] = {};
  int groups = 2;                                 // measured at C2 x 128: 1 stream 1.37 ms, 2 streams 1.31, 4 streams 1.34, 8 streams 1.40
  // CUDA graph of the kernel sequence for small host-buffer batches (launch latency dominates there); re-captured when
  // the shape, the parameters or an option change
  bool use_graph = true;
  cudaGraphExec_t gexec = nullptr;
  int g_B = -1, g_S = -1, g_order = -1, g_launches = 0;
  unsigned long long g_version = 0, version = 1;
  std::vector<cudaEvent_t> ev_in, ev_comp;        // per chunk: input landed / results ready
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  DevBuffers buf{};
  float4* own_in = nullptr;
  unsigned char* raw = nullptr;        // PointCloud2 staging: max_points * URF_MAX_POINT_STEP bytes (urf_process_cloud2)
  unsigned char* rawb = nullptr;       // batched record staging (urf_process_cloud2_batch / _xyz): P * rawb_step bytes, first use
  int rawb_step = 0;
  signed char* label8 = nullptr;       // int8 labels (P bytes), allocated when a caller first asks for them
  int* own_label = nullptr;
  float4* pack = nullptr;              // packed output clouds (urf_process_cloud2_packed): 3 * max_points 32-byte records, allocated on first use
  int* packcnt = nullptr;              // [3][tiles] per-tile counts / offsets
  int* packtot = nullptr;              // [4] cloud sizes
  int* h_packtot = nullptr;            // pinned copy
  urf_params params{};
  DevParams dp{};
  int* h_n = nullptr;          // pinned
  // asynchronous enqueues stage their point counts in a ring of pinned rows, each guarded by the event of its H2D copy,
  // so back-to-back enqueues with different counts never overwrite a row whose copy has not run yet
  static constexpr int kNRing = 8;
  int* h_nring = nullptr;      // pinned, [kNRing][max_batch]
  cudaEvent_t ev_nring[kNRing] = {};
  int nring_pos = 0;
  ScanOut* h_out = nullptr;    // pinned
  int last_B = 0, last_S = 0;
  int launches = 0;
  float last_ms = 0.f;
  bool timing_valid = false;
  std::string err;
  std::vector<void*> allocs;
  // optional per-kernel CUDA-event timing (urf_set_option(ctx, 1, 1)); events live on the ctx stream
  bool profile = false;
  int kslots = 1, kslot = 0;           // event slots: consecutive calls cycle through them so K steps can be timed without syncing
  std::vector<cudaEvent_t> kev;        // [kslots][kMaxKernels + 1]; the last event of a slot closes the pipeline
  std::vector<const char*> knames;
  std::vector<int> kcounts;            // kernels recorded per slot
  int kcount = 0;
};

namespace {

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                               \
      return e_ == cudaErrorMemoryAllocation ? URF_ERR_NOMEM : URF_ERR_CUDA;                        \
    }                                                                                              \
  } while (0)

template <class T> int dalloc(urf_ctx* ctx, T** p, size_t count) {
  void* q = nullptr;
  CK(cudaMalloc(&q, count * sizeof(T) + 256));
  ctx->allocs.push_back(q);
  // zero once: a few kernels issue loads ahead of the bound they are checked against (the values are dropped), and slots of
  // a buffer that a call does not fill must read as something defined
  // (on the context's own stream and waited for: the legacy default stream is not ordered against the non-blocking streams
  // that use the buffer next)
  CK(cudaMemsetAsync(q, 0, count * sizeof(T) + 256, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *p = static_cast<T*>(q);
  return URF_OK;
}

__global__ void k_ring32(DevBuffers buf, int* dst, int S) {
  const int b = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < buf.n[b]) dst[(size_t)b * S + i] = max((int)buf.ringid[(size_t)b * S + i], -1);
}

// View of `buf` for the scans from b0 on: every per-scan array, the workspace included, is advanced by b0 scans (S points
// of stride, T histogram rows per scan).
DevBuffers offset_view(const DevBuffers& a, int b0, int S, int T, int channels) {
  DevBuffers v = a;
  const size_t o = (size_t)b0 * S;
  v.in += o; v.label += o; v.order += o; v.n += b0; v.out += b0;
  if (v.label8) v.label8 += o;
  v.alpha_v += o; v.mark += o; v.ringid += o; v.sect += o; v.bpt += o; v.spt += o; v.ssorted += o;
  v.az += o; v.d2 += o; v.baz += o; v.roadlist += o; v.roadcnt += (size_t)b0 * ((S + 31) >> 5); v.sortbuf += 2 * o;
  v.Tf += (size_t)b0 * channels * kTStride; v.Tb += (size_t)b0 * channels * kTStride;
  v.lut += (size_t)b0 * (kElevBins + 1); v.firstidx += (size_t)b0 * (kElevBins + 1);
  v.hist += (size_t)b0 * T * kRingKeys;
  v.cmin += (size_t)b0 * channels * kDegBins; v.cmax += (size_t)b0 * channels * kDegBins;
  v.ne += (size_t)b0 * channels * (kDegBins + 1);
  v.tab += b0;
  return v;
}

constexpr int kMaxKernels = 32;
constexpr int kMarkSingleMax = 300000;   // scans above this many points take the multi-CTA marker search
thread_local std::string g_create_err;

int launch_pipeline(urf_ctx* ctx, const DevBuffers& buf, int B, int S, bool want_order, bool first = true, bool last = true,
                    cudaStream_t st_override = nullptr) {
  DevParams dp = ctx->dp;
  dp.want_order = want_order ? 1 : 0;
  cudaStream_t st = st_override ? st_override : ctx->stream;
  const int T = (S + kChunk - 1) / kChunk;
  if (T > ctx->Tmax) return URF_ERR_CAPACITY;
  int L = 0;
  ctx->kcount = 0;
  const dim3 gpts((S + 255) / 256, B), gchunk((T + kWarpsPerBlock - 1) / kWarpsPerBlock, B);
  // K(name, launch): one kernel launch; with profiling on, an event is recorded in front of it
#define K(name, ...)                                                                         \
  do {                                                                                       \
    if (ctx->profile && ctx->kcount < kMaxKernels) {                                         \
      ctx->knames[ctx->kcount] = name;                                                       \
      CK(cudaEventRecord(ctx->kev[(size_t)ctx->kslot * (kMaxKernels + 1) + ctx->kcount], st)); \
      ctx->kcount++;                                                                         \
    }                                                                                        \
    __VA_ARGS__;                                                                             \
    L++;                                                                                     \
  } while (0)
  if (first) CK(cudaEventRecord(ctx->ev0, st));
  K("k_reset", k_reset<<<dim3(8, B), 256, 0, st>>>(buf, dp));
  K("k_points", k_points<<<gpts, 256, 0, st>>>(buf, dp, S));
  K("k_register", k_register<<<B, 256, 0, st>>>(buf, dp, S));
  K("k_assign", k_assign<<<gchunk, kWarpsPerBlock * 32, 0, st>>>(buf, dp, S, T));
  K("k_scan_offsets", k_scan_offsets<<<B, 1024, 0, st>>>(buf, dp, S, T));   // + exact re-registration of refuted scans
  K("k_scatter", k_scatter<<<gchunk, kWarpsPerBlock * 32, 0, st>>>(buf, dp, S, T));   // 64 registers, 4 CTAs/SM (48 / 40 registers spill: measured slower)
  // the ring detector next to the star-shaped search: both only read what k_scatter left and add curb hits (idempotent
  // marks, atomic min / max aggregates); k_tab1 is the first reader of the aggregates
  const bool fork = dp.star && !ctx->profile;
  cudaStream_t st_ring = st;
  int side = urf_ctx::kGroups;
  if (fork) {
    for (int g = 0; g < urf_ctx::kGroups; g++) if (st == ctx->s_grp[g]) side = g;
    st_ring = ctx->s_side[side];
    CK(cudaEventRecord(ctx->ev_sfork[side], st));
    CK(cudaStreamWaitEvent(st_ring, ctx->ev_sfork[side], 0));
  }
  const dim3 gtile((S + kTile4 - 1) / kTile4, B);
  {
    cudaStream_t st_main = st;
    st = st_ring;
    if (dp.curbPoints == 5) K("k_ring_detect4", k_ring_detect4<<<gtile, 256, 0, st>>>(buf, dp, S));   // four positions per thread
    else K("k_ring_detect", k_ring_detect<<<gpts, 256, 0, st>>>(buf, dp, S));                        // one position per thread
    st = st_main;
  }
  if (fork) CK(cudaEventRecord(ctx->ev_sjoin[side], st_ring));
  if (dp.star) {
    const int gbig = std::max(4, std::min(kSectKeys, 2048 / B));
    const dim3 gscan((kSectKeys + kScanWarps * 32 - 1) / (kScanWarps * 32), B);
    K("k_star_sort_warp", k_star_sort_warp<<<dim3(kSectKeys, B), 32, 0, st>>>(buf, dp, S));
    K("k_star_sort_big", k_star_sort_big<<<dim3(gbig, B), 256, kStarCtaSmem, st>>>(buf, dp, S));
    K("k_star_scan", k_star_scan<<<gscan, kScanWarps * 32, 0, st>>>(buf, dp, S));
    if (dp.star_prefix)            // sectors whose edge search ran off the near-first prefix: full sort, search resumed
      K("k_star_refine", k_star_refine<<<dim3(std::max(8, std::min(kSectKeys / 8, 8192 / B)), B), 256, kStarCtaSmem, st>>>(buf, dp, S));
  }
  if (fork) CK(cudaStreamWaitEvent(st, ctx->ev_sjoin[side], 0));
  K("k_tab1", k_tab1<<<dim3((dp.channels + 7) / 8, B), 256, 0, st>>>(buf, dp));
  K("k_reach", k_reach<<<dim3((2 * kDegBins + 7) / 8, B), 256, 0, st>>>(buf, dp));
  K("k_tab2", k_tab2<<<dim3((dp.channels + kTab2Rings - 1) / kTab2Rings, B), kTab2Rings * 64, 0, st>>>(buf, dp));
  K("k_label", k_label<<<gpts, 256, 0, st>>>(buf, dp, S));
  if (S <= kMarkSingleMax) K("k_markers1", k_markers1<<<dim3(1, B), kMark1Threads, 0, st>>>(buf, S));   // one CTA per scan
  else {                                                      // large scans: a grid of CTAs per scan, three launches
    const dim3 gm(std::max(1, std::min(64, S / 16384)), B);
    K("k_markers_grid1", k_markers_grid<1><<<gm, kMarkGridThreads, 0, st>>>(buf, S));
    K("k_markers_grid2", k_markers_grid<2><<<gm, kMarkGridThreads, 0, st>>>(buf, S));
    K("k_verts", k_verts<<<B, 384, 0, st>>>(buf, S));
  }
  if (want_order) K("k_sort_rings", k_sort_rings<<<dim3(dp.channels, B), kSortThreads, kRingSmemKeys * sizeof(unsigned long long), st>>>(buf, S));
#undef K
  if (last) CK(cudaEventRecord(ctx->ev1, st));
  if (ctx->profile) {
    CK(cudaEventRecord(ctx->kev[(size_t)ctx->kslot * (kMaxKernels + 1) + kMaxKernels], st));
    ctx->kcounts[ctx->kslot] = ctx->kcount;
    ctx->kslot = (ctx->kslot + 1) % ctx->kslots;
  }
  CK(cudaGetLastError());
  ctx->launches = (first || st_override) ? L : ctx->launches + L;
  ctx->timing_valid = true;
  return URF_OK;
}

// Small batches: replay the whole kernel sequence as one CUDA graph (buf must be ctx->buf itself: constant pointers).
int launch_pipeline_graphed(urf_ctx* ctx, int B, int S, bool want_order) {
  if (!ctx->use_graph || ctx->profile) return launch_pipeline(ctx, ctx->buf, B, S, want_order);
  cudaStream_t st = ctx->stream;
  if (!ctx->gexec || ctx->g_B != B || ctx->g_S != S || ctx->g_order != (int)want_order || ctx->g_version != ctx->version) {
    if (ctx->gexec) { cudaGraphExecDestroy(ctx->gexec); ctx->gexec = nullptr; }
    cudaGraph_t graph = nullptr;
    CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    ctx->launches = 0;
    const int rc = launch_pipeline(ctx, ctx->buf, B, S, want_order, false, false);
    const cudaError_t e = cudaStreamEndCapture(st, &graph);
    if (rc != URF_OK || e != cudaSuccess || !graph) { if (graph) cudaGraphDestroy(graph); ctx->err = "graph capture failed"; return rc != URF_OK ? rc : URF_ERR_CUDA; }
    const cudaError_t ei = cudaGraphInstantiate(&ctx->gexec, graph, 0);
    cudaGraphDestroy(graph);
    if (ei != cudaSuccess) { ctx->gexec = nullptr; ctx->err = cudaGetErrorString(ei); return URF_ERR_CUDA; }
    ctx->g_B = B; ctx->g_S = S; ctx->g_order = (int)want_order; ctx->g_version = ctx->version; ctx->g_launches = ctx->launches;
  }
  CK(cudaEventRecord(ctx->ev0, st));
  CK(cudaGraphLaunch(ctx->gexec, st));
  CK(cudaEventRecord(ctx->ev1, st));
  ctx->launches = ctx->g_launches;
  ctx->timing_valid = true;
  return URF_OK;
}

void fill_result(const ScanOut& o, urf_result* r) {
  r->n_in = o.n_in; r->n_roi = o.n_roi;
  r->flags = o.flags & F_PUBLIC_MASK; r->reserved = 0;
  if (o.n_roi < 30) {                       // lidar_segmentation.cpp:124-126
    r->status = URF_TOO_FEW_POINTS;
    r->n_rings = 0; r->n_order = 0; r->n_road = 0; r->n_curb = 0; r->n_vert = 0;
    if (r->ring_start) for (int k = 0; k <= URF_MAX_CHANNELS; k++) r->ring_start[k] = 0;
    return;
  }
  r->status = URF_OK;
  r->n_rings = o.n_rings; r->n_order = o.n_order; r->n_road = o.n_road; r->n_curb = o.n_curb; r->n_vert = o.n_vert;
  std::memcpy(r->vert, o.vert, sizeof(float) * 4 * (size_t)o.n_vert);
  if (r->ring_start) std::memcpy(r->ring_start, o.ring_start, sizeof(int) * (URF_MAX_CHANNELS + 1));
}

}  // namespace

extern "C" {

int urf_version(void) { return URF_VERSION; }

const char* urf_strerror(int code) {
  switch (code) {
    case URF_OK: return "ok";
    case URF_TOO_FEW_POINTS: return "fewer than 30 points in the ROI: nothing published";
    case URF_ERR_INVALID: return "invalid argument";
    case URF_ERR_NO_DEVICE: return "no CUDA device (this library has no CPU fallback)";
    case URF_ERR_CUDA: return "CUDA error";
    case URF_ERR_NOMEM: return "out of device or pinned memory";
    case URF_ERR_CAPACITY: return "scan or batch larger than the context was created for";
    case URF_ERR_TIMEOUT: return "timed out";
    case URF_ERR_CLOSED: return "queue closed";
    default: return "unknown error";
  }
}

const char* urf_last_cuda_error(const urf_ctx* ctx) {
  if (ctx) return ctx->err.c_str();
  return g_create_err.empty() ? "null context" : g_create_err.c_str();     // text of this thread's last failed urf_create
}

void urf_default_params(urf_params* p) {
  if (!p) return;
  std::memset(p, 0, sizeof(*p));
  std::snprintf(p->fixed_frame, sizeof(p->fixed_frame), "left_os1/os1_lidar");
  std::snprintf(p->topic_name, sizeof(p->topic_name), "/left_os1/os1_cloud_node/points");
  p->x_zero_method = 1; p->z_zero_method = 1; p->star_shaped_method = 1; p->blind_spots = 1; p->xDirection = 0;
  p->interval = 0.18; p->curb_height = 0.05; p->curb_points = 5; p->beamZone = 30;
  p->min_x = 0; p->max_x = 30; p->min_y = -10; p->max_y = 10; p->min_z = -3; p->max_z = -1;
  p->cylinder_deg_x = 150; p->cylinder_deg_z = 140; p->curb_slope_deg = 50;
  p->kdev_param = 1.225; p->kdist_param = 2; p->starbeam_filter = 0; p->dmin_param = 10;
  p->simple_poly_allow = 1; p->poly_s_param = 0.7; p->poly_z_manual = -1.5; p->poly_z_avg_allow = 1;
  p->channels = 64;
}

int urf_create(urf_ctx** out, int device, int max_points, int max_batch) {
  if (!out || max_points < 1 || max_batch < 1 || max_points > (1 << 24)) return URF_ERR_INVALID;
  if ((long long)(max_points + kChunk) * max_batch >= (1ll << 31)) return URF_ERR_CAPACITY;   // kernels use 32-bit offsets
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return URF_ERR_NO_DEVICE;
  urf_ctx* ctx = new urf_ctx();
  // the context dies with the failure: its error text survives in a per-thread slot that urf_last_cuda_error(NULL) returns
  auto fail = [&](int rc) { g_create_err = ctx->err.empty() ? std::string(urf_strerror(rc)) : ctx->err; urf_destroy(ctx); return rc; };
  ctx->device = device;
  if (cudaSetDevice(device) != cudaSuccess) return fail(URF_ERR_NO_DEVICE);
  ctx->max_points = ((max_points + kChunk - 1) / kChunk) * kChunk;
  ctx->max_batch = max_batch;
  ctx->P = (size_t)ctx->max_points * max_batch;
  ctx->Tmax = ctx->max_points / kChunk;
  int rc;
#define TRY(x) do { rc = (x); if (rc != URF_OK) return fail(rc); } while (0)
#define CKF(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { ctx->err = cudaGetErrorString(e_); return fail(URF_ERR_CUDA); } } while (0)
  CKF(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  CKF(cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking));
  CKF(cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking));
  for (int g = 0; g < urf_ctx::kGroups; g++) {
    CKF(cudaStreamCreateWithFlags(&ctx->s_grp[g], cudaStreamNonBlocking));
    CKF(cudaEventCreateWithFlags(&ctx->ev_join[g], cudaEventDisableTiming));
  }
  CKF(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
  for (int g = 0; g <= urf_ctx::kGroups; g++) {
    CKF(cudaStreamCreateWithFlags(&ctx->s_side[g], cudaStreamNonBlocking));
    CKF(cudaEventCreateWithFlags(&ctx->ev_sfork[g], cudaEventDisableTiming));
    CKF(cudaEventCreateWithFlags(&ctx->ev_sjoin[g], cudaEventDisableTiming));
  }
  CKF(cudaEventCreate(&ctx->ev0));
  CKF(cudaEventCreate(&ctx->ev1));
  const size_t P = ctx->P;
  DevBuffers& b = ctx->buf;
  TRY(dalloc(ctx, &ctx->own_in, P));
  TRY(dalloc(ctx, &ctx->raw, (size_t)ctx->max_points * URF_MAX_POINT_STEP));
  TRY(dalloc(ctx, &b.alpha_v, P));
  TRY(dalloc(ctx, &b.mark, P));
  TRY(dalloc(ctx, &b.ringid, P));
  TRY(dalloc(ctx, &b.sect, P));
  TRY(dalloc(ctx, &ctx->own_label, P));
  TRY(dalloc(ctx, &b.bpt, P));
  TRY(dalloc(ctx, &b.spt, P));
  TRY(dalloc(ctx, &b.ssorted, P));
  TRY(dalloc(ctx, &b.az, P));
  TRY(dalloc(ctx, &b.d2, P));
  TRY(dalloc(ctx, &b.baz, P));
  TRY(dalloc(ctx, &b.roadlist, P));
  TRY(dalloc(ctx, &b.roadcnt, P / 32 + (size_t)max_batch + 1));
  TRY(dalloc(ctx, &b.Tf, (size_t)max_batch * kTStride * URF_MAX_CHANNELS));
  TRY(dalloc(ctx, &b.Tb, (size_t)max_batch * kTStride * URF_MAX_CHANNELS));
  TRY(dalloc(ctx, &b.lut, (size_t)max_batch * (kElevBins + 1)));
  TRY(dalloc(ctx, &b.order, P));
  TRY(dalloc(ctx, &b.sortbuf, 2 * P));
  TRY(dalloc(ctx, &b.hist, (size_t)max_batch * ctx->Tmax * kRingKeys));
  TRY(dalloc(ctx, &b.firstidx, (size_t)max_batch * (kElevBins + 1)));
  TRY(dalloc(ctx, &b.cmin, (size_t)max_batch * URF_MAX_CHANNELS * kDegBins));
  TRY(dalloc(ctx, &b.cmax, (size_t)max_batch * URF_MAX_CHANNELS * kDegBins));
  TRY(dalloc(ctx, &b.ne, (size_t)max_batch * URF_MAX_CHANNELS * (kDegBins + 1)));
  TRY(dalloc(ctx, &b.newY, (size_t)ctx->max_points));
  TRY(dalloc(ctx, &b.n, (size_t)max_batch));
  TRY(dalloc(ctx, &b.out, (size_t)max_batch));
  TRY(dalloc(ctx, &b.tab, (size_t)max_batch));
  b.in = ctx->own_in;
  b.label = ctx->own_label;
  CKF(cudaMallocHost((void**)&ctx->h_n, sizeof(int) * max_batch));
  CKF(cudaMallocHost((void**)&ctx->h_nring, sizeof(int) * max_batch * urf_ctx::kNRing));
  for (int r = 0; r < urf_ctx::kNRing; r++) CKF(cudaEventCreateWithFlags(&ctx->ev_nring[r], cudaEventDisableTiming));
  CKF(cudaMallocHost((void**)&ctx->h_out, sizeof(ScanOut) * max_batch));
  {
    std::vector<float> ny;
    host_newY(ny, ctx->max_points);
    CKF(cudaMemcpy(b.newY, ny.data(), sizeof(float) * ny.size(), cudaMemcpyHostToDevice));
    float bd[kSectKeys], bo[kSectKeys], Kfi;
    unsigned char byx[kSectKeys];
    host_beam_init(bd, bo, byx, &Kfi);
    CKF(cudaMemcpyToSymbol(c_beam_d, bd, sizeof(bd)));
    CKF(cudaMemcpyToSymbol(c_beam_o, bo, sizeof(bo)));
    CKF(cudaMemcpyToSymbol(c_beam_yx, byx, sizeof(byx)));
    ctx->dp.Kfi = Kfi;
  }
  CKF(cudaFuncSetAttribute(k_star_sort_big, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kStarCtaSmem));
  CKF(cudaFuncSetAttribute(k_star_refine, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kStarCtaSmem));
  CKF(cudaFuncSetAttribute(k_sort_rings, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kRingSmemKeys * sizeof(unsigned long long))));
  urf_default_params(&ctx->params);
  narrow_params(&ctx->params, &ctx->dp, ctx->dp.Kfi, 0, 0);
  ctx->dp.star_prefix = 1;                                  // near-first star sort
#undef TRY
#undef CKF
  *out = ctx;
  return URF_OK;
}

void urf_destroy(urf_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  for (void* p : ctx->allocs) cudaFree(p);
  if (ctx->h_n) cudaFreeHost(ctx->h_n);
  if (ctx->h_nring) cudaFreeHost(ctx->h_nring);
  for (cudaEvent_t e : ctx->ev_nring) if (e) cudaEventDestroy(e);
  if (ctx->h_out) cudaFreeHost(ctx->h_out);
  if (ctx->h_packtot) cudaFreeHost(ctx->h_packtot);
  if (ctx->gexec) cudaGraphExecDestroy(ctx->gexec);
  for (cudaEvent_t e : ctx->kev) cudaEventDestroy(e);
  for (cudaEvent_t e : ctx->ev_in) cudaEventDestroy(e);
  for (cudaEvent_t e : ctx->ev_comp) cudaEventDestroy(e);
  for (int g = 0; g < urf_ctx::kGroups; g++) { if (ctx->s_grp[g]) cudaStreamDestroy(ctx->s_grp[g]); if (ctx->ev_join[g]) cudaEventDestroy(ctx->ev_join[g]); }
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  for (int g = 0; g <= urf_ctx::kGroups; g++) {
    if (ctx->s_side[g]) cudaStreamDestroy(ctx->s_side[g]);
    if (ctx->ev_sfork[g]) cudaEventDestroy(ctx->ev_sfork[g]);
    if (ctx->ev_sjoin[g]) cudaEventDestroy(ctx->ev_sjoin[g]);
  }
  if (ctx->s_in) cudaStreamDestroy(ctx->s_in);
  if (ctx->s_out) cudaStreamDestroy(ctx->s_out);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

void* urf_pinned_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return p;
}
void urf_pinned_free(void* p) { if (p) cudaFreeHost(p); }

int urf_set_params(urf_ctx* ctx, const urf_params* p) {
  if (!ctx || !p) return URF_ERR_INVALID;
  int rc = validate_params(p);
  if (rc != URF_OK) return rc;
  ctx->params = *p;
  narrow_params(p, &ctx->dp, ctx->dp.Kfi, ctx->dp.force_exact, 0);
  ctx->version++;
  return URF_OK;
}

int urf_get_params(const urf_ctx* ctx, urf_params* p) {
  if (!ctx || !p) return URF_ERR_INVALID;
  *p = ctx->params;
  return URF_OK;
}

// test/diagnostic options: 0 = force exact ring registration (0/1); 1 = per-kernel CUDA-event timing (slots, 0 = off);
// 2 = number of compute streams a device-resident batch is spread over (1..16); 3 = CUDA graph for small batches (0/1);
// 4 = near-first star sort (0/1, default 1).
// Options 5-12 selected tuning variants that were measured slower and removed (DESIGN.md §6). Each still accepts the
// value that is now built in, so existing settings keep working, and rejects any other value:
// 5 scans per sub-batch (0 = batch / streams), 6 batch CUDA graph (0), 7 shared workspace slot (0), 8 ring detector
// (46: k_ring_detect4 at 6 CTAs/SM for curb_points 5, else k_ring_detect), 9 marker search (1: one CTA per scan up to
// kMarkSingleMax points, else a grid), 10 near-first pivot rank (kStarPivot), 11 ring detector on a side stream (1),
// 12 widest single-warp star sort network (16 elements per lane).
int urf_set_option(urf_ctx* ctx, int option, int value) {
  if (!ctx) return URF_ERR_INVALID;
  static constexpr int kRetired[][2] = {{5, 0}, {6, 0}, {7, 0}, {8, 46}, {9, 1}, {10, kStarPivot}, {11, 1}, {12, 16}};
  for (const auto& r : kRetired)
    if (option == r[0]) return value == r[1] ? URF_OK : URF_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  ctx->version++;
  if (option == 0) { ctx->dp.force_exact = value != 0; ctx->version++; return URF_OK; }
  if (option == 4) { ctx->dp.star_prefix = value != 0; ctx->version++; return URF_OK; }
  if (option == 3) { ctx->use_graph = value != 0; return URF_OK; }
  if (option == 2) { ctx->groups = value < 1 ? 1 : (value > urf_ctx::kGroups ? urf_ctx::kGroups : value); return URF_OK; }
  if (option == 1) {                   // value = number of event slots (0 = off)
    CK(cudaStreamSynchronize(ctx->stream));               // events of the previous setting may still be pending
    if (ctx->gexec) { cudaGraphExecDestroy(ctx->gexec); ctx->gexec = nullptr; ctx->g_B = -1; }
    for (cudaEvent_t e : ctx->kev) cudaEventDestroy(e);
    ctx->kev.clear();
    ctx->profile = value > 0;
    ctx->kslots = value > 0 ? value : 1;
    ctx->kslot = 0;
    if (ctx->profile) {
      ctx->kev.assign((size_t)ctx->kslots * (kMaxKernels + 1), nullptr);
      for (cudaEvent_t& e : ctx->kev) {
        const cudaError_t ce = cudaEventCreate(&e);
        if (ce != cudaSuccess) {                           // leave the option off and leak nothing
          for (cudaEvent_t f : ctx->kev) if (f) cudaEventDestroy(f);
          ctx->kev.clear(); ctx->profile = false; ctx->kslots = 1;
          ctx->err = std::string("cudaEventCreate: ") + cudaGetErrorString(ce);
          return URF_ERR_CUDA;
        }
      }
      ctx->knames.assign(kMaxKernels, "");
      ctx->kcounts.assign(ctx->kslots, 0);
    }
    return URF_OK;
  }
  return URF_ERR_INVALID;
}

void* urf_stream(urf_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

float urf_last_device_ms(const urf_ctx* c) {
  urf_ctx* ctx = const_cast<urf_ctx*>(c);
  if (!ctx || !ctx->timing_valid) return -1.f;
  float ms = -1.f;
  if (cudaEventSynchronize(ctx->ev1) != cudaSuccess) return -1.f;
  if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) != cudaSuccess) return -1.f;
  return ms;
}

int urf_last_launch_count(const urf_ctx* ctx) { return ctx ? ctx->launches : 0; }

// With option 1 on: number of kernels of the last call, and name / device milliseconds of kernel `idx` (event before it to
// the event before the next kernel, or to the end-of-pipeline event for the last one). Waits for the stream.
int urf_profile_count(const urf_ctx* ctx) { return ctx && ctx->profile ? ctx->kcounts[0] : 0; }
int urf_profile_slots(const urf_ctx* ctx) { return ctx && ctx->profile ? ctx->kslots : 0; }
// name / device milliseconds of kernel `idx` in event slot `slot` (the slot's calls must have completed)
int urf_profile_get(urf_ctx* ctx, int slot, int idx, const char** name, float* ms) {
  if (!ctx || !ctx->profile || slot < 0 || slot >= ctx->kslots || idx < 0 || idx >= ctx->kcounts[slot]) return URF_ERR_INVALID;
  const size_t o = (size_t)slot * (kMaxKernels + 1);
  cudaEvent_t next = idx + 1 < ctx->kcounts[slot] ? ctx->kev[o + idx + 1] : ctx->kev[o + kMaxKernels];
  CK(cudaEventSynchronize(next));
  CK(cudaEventElapsedTime(ms, ctx->kev[o + idx], next));
  if (name) *name = ctx->knames[idx];
  return URF_OK;
}

int urf_enqueue_batch_device_ex(urf_ctx* ctx, const float* d_xyzi, int stride_points, const int* n, int batch, int32_t* d_label,
                                int32_t* d_order) {
  if (!ctx || !d_xyzi || !n || !d_label || batch < 1 || stride_points < 1) return URF_ERR_INVALID;
  if (batch > ctx->max_batch || (size_t)stride_points * batch > ctx->P || stride_points > ctx->max_points) return URF_ERR_CAPACITY;
  CK(cudaSetDevice(ctx->device));
  for (int b = 0; b < batch; b++) if (n[b] < 0 || n[b] > stride_points) return URF_ERR_INVALID;
  int* row = ctx->h_nring + (size_t)ctx->nring_pos * ctx->max_batch;
  CK(cudaEventSynchronize(ctx->ev_nring[ctx->nring_pos]));    // the copy that last used this row (kNRing enqueues ago) is done
  std::memcpy(row, n, sizeof(int) * batch);
  CK(cudaMemcpyAsync(ctx->buf.n, row, sizeof(int) * batch, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaEventRecord(ctx->ev_nring[ctx->nring_pos], ctx->stream));
  ctx->nring_pos = (ctx->nring_pos + 1) % urf_ctx::kNRing;
  const bool want_order = d_order != nullptr;
  DevBuffers bufv = ctx->buf;                                 // the caller's buffers instead of the context's own
  bufv.in = reinterpret_cast<float4*>(const_cast<float*>(d_xyzi));
  bufv.label = d_label;
  if (want_order) bufv.order = d_order;
  int rc = URF_OK;
  const int T = (stride_points + kChunk - 1) / kChunk;
  const int sub = (batch + ctx->groups - 1) / ctx->groups;    // scans per stream
  const int G = (ctx->profile || batch < 2 * ctx->groups) ? 1 : (batch + sub - 1) / sub;   // per-kernel event timing needs one stream
  if (G == 1) rc = launch_pipeline(ctx, bufv, batch, stride_points, want_order);
  else {
    // fork: the ctx stream hands one sub-batch to each group stream and joins them again, so callers still see ONE stream
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    CK(cudaEventRecord(ctx->ev_fork, ctx->stream));
    int launches = 0;
    for (int g = 0; g < G; g++) {
      const int b0 = g * sub;
      CK(cudaStreamWaitEvent(ctx->s_grp[g], ctx->ev_fork, 0));
      rc = launch_pipeline(ctx, offset_view(bufv, b0, stride_points, T, ctx->dp.channels), std::min(sub, batch - b0), stride_points,
                           want_order, false, false, ctx->s_grp[g]);
      if (rc != URF_OK) break;
      launches += ctx->launches;
    }
    for (int g = 0; g < G; g++) {
      CK(cudaEventRecord(ctx->ev_join[g], ctx->s_grp[g]));
      CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[g], 0));
    }
    ctx->launches = launches;
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
  }
  ctx->last_B = batch; ctx->last_S = stride_points;
  return rc;
}

int urf_enqueue_batch_device(urf_ctx* ctx, const float* d_xyzi, int stride_points, const int* n, int batch, int32_t* d_label) {
  return urf_enqueue_batch_device_ex(ctx, d_xyzi, stride_points, n, batch, d_label, nullptr);
}

int urf_finish_batch_device(urf_ctx* ctx, urf_result* outs) {
  if (!ctx) return URF_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  const int B = ctx->last_B;
  if (outs) CK(cudaMemcpyAsync(ctx->h_out, ctx->buf.out, sizeof(ScanOut) * B, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (outs) for (int b = 0; b < B; b++) {
    urf_result tmp = outs[b];
    tmp.ring_start = nullptr;
    fill_result(ctx->h_out[b], &tmp);
    tmp.label = outs[b].label; tmp.ring = outs[b].ring; tmp.order = outs[b].order; tmp.ring_start = outs[b].ring_start;
    outs[b] = tmp;
  }
  return URF_OK;
}

int urf_process_batch_device(urf_ctx* ctx, const float* d_xyzi, int stride_points, const int* n, int batch,
                             int32_t* d_label, urf_result* outs) {
  int rc = urf_enqueue_batch_device(ctx, d_xyzi, stride_points, n, batch, d_label);
  if (rc != URF_OK) return rc;
  return urf_finish_batch_device(ctx, outs);
}

namespace {
// Shared body of the host-buffer batch entry points. step == 0: data[b] holds n[b] (x, y, z, intensity) float4 records that
// are copied straight into the input buffer; step > 0: data[b] holds n[b] records of `step` bytes with FLOAT32 x / y / z /
// intensity at the given byte offsets (oi < 0: none) — the raw bytes cross PCIe and are unpacked on the device.
// label8 (or NULL): per scan an int8 HOST buffer for the labels (one byte per point instead of four).
int process_batch_impl(urf_ctx* ctx, const void* const* data, const int* n, int batch, int step, int ox, int oy, int oz, int oi,
                       urf_result* outs, int8_t* const* label8) {
  if (!ctx || !data || !n || !outs || batch < 1) return URF_ERR_INVALID;
  if (batch > ctx->max_batch) return URF_ERR_CAPACITY;
  if (step != 0) {
    if (step < 12 || step > URF_MAX_POINT_STEP) return URF_ERR_INVALID;
    for (int o : {ox, oy, oz}) if (o < 0 || o + 4 > step) return URF_ERR_INVALID;
    if (oi >= 0 && oi + 4 > step) return URF_ERR_INVALID;
  }
  CK(cudaSetDevice(ctx->device));
  int nmax = 1;
  bool want_order = false, want_ring = false, want_l8 = false;
  for (int b = 0; b < batch; b++) {
    if (n[b] < 0 || (n[b] > 0 && !data[b])) return URF_ERR_INVALID;
    if (n[b] > ctx->max_points) return URF_ERR_CAPACITY;
    nmax = n[b] > nmax ? n[b] : nmax;
    want_order |= outs[b].order != nullptr;
    want_ring |= outs[b].ring != nullptr;
    want_l8 |= label8 && label8[b];
    ctx->h_n[b] = n[b];
  }
  if (step != 0 && (!ctx->rawb || ctx->rawb_step < step)) {      // first use (or a wider record than before): P * step bytes
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->rawb) { cudaFree(ctx->rawb); ctx->allocs.erase(std::find(ctx->allocs.begin(), ctx->allocs.end(), (void*)ctx->rawb)); ctx->rawb = nullptr; }
    const int rc = dalloc(ctx, &ctx->rawb, ctx->P * (size_t)step);
    if (rc != URF_OK) return rc;
    ctx->rawb_step = step;
  }
  if (want_l8 && !ctx->label8) {
    const int rc = dalloc(ctx, &ctx->label8, ctx->P);
    if (rc != URF_OK) return rc;
  }
  const int S = ((nmax + 255) / 256) * 256;
  const int T = (S + kChunk - 1) / kChunk;
  cudaStream_t st = ctx->stream;
  DevBuffers bufv = ctx->buf;
  bufv.label8 = want_l8 ? ctx->label8 : nullptr;
  // Software pipeline over chunks of scans: H2D of chunk c+1 (s_in), kernels of chunk c (stream) and D2H of chunk c-1
  // (s_out) overlap; scans are independent, every chunk owns its slice of every buffer.
  // Chunks of batch / 16 scans. (Measured and dropped: smaller chunks at both ends of the call — a shorter pipeline fill and
  // drain on paper, 5 % slower in practice — and copies running only three chunks ahead of the launches.)
  std::vector<int> cb;                                        // chunk c = scans [cb[c], cb[c + 1])
  {
    const int chunk = batch >= 16 ? std::max(4, (batch + 15) / 16) : batch;
    for (int b0 = 0; b0 < batch; b0 += chunk) cb.push_back(b0);
    cb.push_back(batch);
  }
  const int nchunks = (int)cb.size() - 1;
  while ((int)ctx->ev_in.size() < nchunks) {
    cudaEvent_t a, c;
    CK(cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&c, cudaEventDisableTiming));
    ctx->ev_in.push_back(a); ctx->ev_comp.push_back(c);
  }
  int* ring32 = reinterpret_cast<int*>(ctx->buf.sortbuf);     // free once the sorts of a chunk are done (chunk-private slice)
  const bool graphed = nchunks == 1 && batch <= 8 && !want_l8;
  // every host-to-device copy of the call is queued first (the copies depend on nothing): the copy engine then never waits
  // for this thread to get through a chunk's kernel launches and result copies
  for (int c = 0; c < nchunks; c++) {
    const int b0 = cb[c], nb = cb[c + 1] - b0;
    CK(cudaMemcpyAsync(ctx->buf.n + b0, ctx->h_n + b0, sizeof(int) * nb, cudaMemcpyHostToDevice, ctx->s_in));
    for (int b = b0; b < b0 + nb; b++) {
      if (n[b] <= 0) continue;
      if (step == 0) CK(cudaMemcpyAsync(ctx->own_in + (size_t)b * S, data[b], sizeof(float) * 4 * (size_t)n[b], cudaMemcpyHostToDevice, ctx->s_in));
      else CK(cudaMemcpyAsync(ctx->rawb + (size_t)b * S * step, data[b], (size_t)step * (size_t)n[b], cudaMemcpyHostToDevice, ctx->s_in));
    }
    CK(cudaEventRecord(ctx->ev_in[c], ctx->s_in));
  }
  for (int c = 0; c < nchunks; c++) {
    const int b0 = cb[c], nb = cb[c + 1] - b0;
    CK(cudaStreamWaitEvent(st, ctx->ev_in[c], 0));
    if (step != 0)
      k_unpack_cloud2_batch<<<dim3((S + 255) / 256, nb), 256, 0, st>>>(ctx->rawb + (size_t)b0 * S * step, ctx->own_in + (size_t)b0 * S, ctx->buf.n + b0, S,
                                                                          step, ox, oy, oz, oi);
    const DevBuffers view = offset_view(bufv, b0, S, T, ctx->dp.channels);
    int rc = graphed ? launch_pipeline_graphed(ctx, nb, S, want_order) : launch_pipeline(ctx, view, nb, S, want_order, c == 0, c == nchunks - 1);
    if (rc != URF_OK) {                                 // nothing of this call may still be writing into the caller's buffers
      cudaStreamSynchronize(ctx->s_in); cudaStreamSynchronize(st); cudaStreamSynchronize(ctx->s_out);
      return rc;
    }
    if (want_ring) k_ring32<<<dim3((S + 255) / 256, nb), 256, 0, st>>>(view, ring32 + (size_t)b0 * S * 4, S);
    CK(cudaEventRecord(ctx->ev_comp[c], st));
    CK(cudaStreamWaitEvent(ctx->s_out, ctx->ev_comp[c], 0));
    CK(cudaMemcpyAsync(ctx->h_out + b0, ctx->buf.out + b0, sizeof(ScanOut) * nb, cudaMemcpyDeviceToHost, ctx->s_out));
    for (int b = b0; b < b0 + nb; b++) {
      if (n[b] <= 0) continue;
      if (outs[b].label) CK(cudaMemcpyAsync(outs[b].label, ctx->own_label + (size_t)b * S, sizeof(int) * (size_t)n[b], cudaMemcpyDeviceToHost, ctx->s_out));
      if (label8 && label8[b]) CK(cudaMemcpyAsync(label8[b], ctx->label8 + (size_t)b * S, (size_t)n[b], cudaMemcpyDeviceToHost, ctx->s_out));
      if (outs[b].ring) CK(cudaMemcpyAsync(outs[b].ring, ring32 + (size_t)b0 * S * 4 + (size_t)(b - b0) * S, sizeof(int) * (size_t)n[b], cudaMemcpyDeviceToHost, ctx->s_out));
      if (outs[b].order) CK(cudaMemcpyAsync(outs[b].order, ctx->buf.order + (size_t)b * S, sizeof(int) * (size_t)n[b], cudaMemcpyDeviceToHost, ctx->s_out));
    }
  }
  CK(cudaStreamSynchronize(ctx->s_out));
  CK(cudaStreamSynchronize(st));
  ctx->last_B = batch; ctx->last_S = S;
  for (int b = 0; b < batch; b++) {
    fill_result(ctx->h_out[b], &outs[b]);
    if (outs[b].status == URF_TOO_FEW_POINTS && outs[b].ring) for (int i = 0; i < n[b]; i++) outs[b].ring[i] = -1;
  }
  return URF_OK;
}
}  // namespace

int urf_process_batch(urf_ctx* ctx, const float* const* xyzi, const int* n, int batch, urf_result* outs) {
  return process_batch_impl(ctx, reinterpret_cast<const void* const*>(xyzi), n, batch, 0, 0, 0, 0, -1, outs, nullptr);
}

int urf_process_batch_xyz(urf_ctx* ctx, const float* const* xyz, const int* n, int batch, urf_result* outs, int8_t* const* label8) {
  return process_batch_impl(ctx, reinterpret_cast<const void* const*>(xyz), n, batch, 12, 0, 4, 8, -1, outs, label8);
}

int urf_process_cloud2_batch(urf_ctx* ctx, const void* const* data, const int* n_points, int batch, int point_step, int off_x, int off_y,
                             int off_z, int off_intensity, urf_result* outs, int8_t* const* label8) {
  if (point_step == 0) return URF_ERR_INVALID;
  return process_batch_impl(ctx, data, n_points, batch, point_step, off_x, off_y, off_z, off_intensity, outs, label8);
}

namespace {
// Shared body of urf_process_cloud2 / urf_process_cloud2_packed: H2D of the raw records, unpack, pipeline, optional pack.
int process_cloud2(urf_ctx* ctx, const void* data, int n, int point_step, int off_x, int off_y, int off_z, int off_i,
                   urf_result* out, urf_clouds* clouds) {
  if (!ctx || !out || n < 0 || (n > 0 && !data)) return URF_ERR_INVALID;
  if (point_step < 12 || point_step > URF_MAX_POINT_STEP) return URF_ERR_INVALID;
  for (int o : {off_x, off_y, off_z}) if (o < 0 || o + 4 > point_step) return URF_ERR_INVALID;
  if (off_i >= 0 && off_i + 4 > point_step) return URF_ERR_INVALID;
  if (n > ctx->max_points) return URF_ERR_CAPACITY;
  CK(cudaSetDevice(ctx->device));
  const int tiles = (std::max(ctx->max_points, 1) + kPackTile - 1) / kPackTile;
  if (clouds && !ctx->pack) {                                // first packed call: 96 bytes per point of capacity
    int rc = dalloc(ctx, &ctx->pack, (size_t)6 * ctx->max_points);
    if (rc == URF_OK) rc = dalloc(ctx, &ctx->packcnt, (size_t)3 * tiles);
    if (rc == URF_OK) rc = dalloc(ctx, &ctx->packtot, 4);
    if (rc != URF_OK) { ctx->pack = nullptr; return rc; }
    CK(cudaMallocHost((void**)&ctx->h_packtot, sizeof(int) * 4));
  }
  const int S = ((std::max(n, 1) + 255) / 256) * 256;
  cudaStream_t st = ctx->stream;
  ctx->h_n[0] = n;
  CK(cudaMemcpyAsync(ctx->buf.n, ctx->h_n, sizeof(int), cudaMemcpyHostToDevice, st));
  if (n > 0) {
    CK(cudaMemcpyAsync(ctx->raw, data, (size_t)n * point_step, cudaMemcpyHostToDevice, st));
    k_unpack_cloud2<<<(n + 255) / 256, 256, 0, st>>>(ctx->raw, ctx->own_in, n, point_step, off_x, off_y, off_z, off_i);
  }
  const bool want_order = out->order != nullptr || clouds != nullptr;
  int rc = launch_pipeline_graphed(ctx, 1, S, want_order);
  if (rc != URF_OK) return rc;
  int* ring32 = reinterpret_cast<int*>(ctx->buf.sortbuf);
  if (out->ring) k_ring32<<<dim3((S + 255) / 256, 1), 256, 0, st>>>(ctx->buf, ring32, S);
  float4 *d_rc = nullptr, *d_roi = nullptr, *d_prob = nullptr;
  if (clouds) {
    const int nt = (std::max(n, 1) + kPackTile - 1) / kPackTile;
    d_rc = ctx->pack; d_roi = ctx->pack + 2 * (size_t)ctx->max_points; d_prob = ctx->pack + 4 * (size_t)ctx->max_points;
    k_pack_count<<<nt, 256, 0, st>>>(ctx->buf, ctx->packcnt, nt);
    k_pack_scan<<<1, 1024, 0, st>>>(ctx->buf, ctx->packcnt, nt, ctx->packtot);
    k_pack_write<<<nt, 256, 0, st>>>(ctx->buf, ctx->packcnt, nt, ctx->packtot, d_rc, d_roi, d_prob);
    ctx->launches += 3;
    CK(cudaMemcpyAsync(ctx->h_packtot, ctx->packtot, sizeof(int) * 4, cudaMemcpyDeviceToHost, st));
  }
  CK(cudaMemcpyAsync(ctx->h_out, ctx->buf.out, sizeof(ScanOut), cudaMemcpyDeviceToHost, st));
  if (n > 0) {
    if (out->label) CK(cudaMemcpyAsync(out->label, ctx->own_label, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, st));
    if (out->ring) CK(cudaMemcpyAsync(out->ring, ring32, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, st));
    if (out->order) CK(cudaMemcpyAsync(out->order, ctx->buf.order, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, st));
  }
  CK(cudaStreamSynchronize(st));
  if (clouds) {                                              // sizes are known now: copy exactly the records that exist
    const int* t = ctx->h_packtot;
    clouds->n_road = t[0]; clouds->n_curb = t[1]; clouds->n_roi = t[2]; clouds->n_road_probably = t[3];
    const size_t rec = sizeof(urf_point_xyzi);
    if (clouds->road && t[0] > 0) CK(cudaMemcpyAsync(clouds->road, d_rc, rec * t[0], cudaMemcpyDeviceToHost, st));
    if (clouds->curb && t[1] > 0) CK(cudaMemcpyAsync(clouds->curb, d_rc + 2 * (size_t)t[0], rec * t[1], cudaMemcpyDeviceToHost, st));
    if (clouds->roi && t[2] > 0) CK(cudaMemcpyAsync(clouds->roi, d_roi, rec * t[2], cudaMemcpyDeviceToHost, st));
    if (clouds->road_probably && t[3] > 0) CK(cudaMemcpyAsync(clouds->road_probably, d_prob, rec * t[3], cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  ctx->last_B = 1; ctx->last_S = S;
  fill_result(ctx->h_out[0], out);
  if (out->status == URF_TOO_FEW_POINTS && out->ring) for (int i = 0; i < n; i++) out->ring[i] = -1;
  return URF_OK;
}
}  // namespace

int urf_process_cloud2(urf_ctx* ctx, const void* data, int n, int point_step, int off_x, int off_y, int off_z, urf_result* out) {
  return process_cloud2(ctx, data, n, point_step, off_x, off_y, off_z, -1, out, nullptr);
}

int urf_process_cloud2_packed(urf_ctx* ctx, const void* data, int n, int point_step, int off_x, int off_y, int off_z,
                              int off_intensity, urf_result* out, urf_clouds* clouds) {
  if (!clouds) return URF_ERR_INVALID;
  return process_cloud2(ctx, data, n, point_step, off_x, off_y, off_z, off_intensity, out, clouds);
}

int urf_process(urf_ctx* ctx, const float* xyzi, int n, urf_result* out) {
  const float* ptrs[1] = {xyzi};
  return urf_process_batch(ctx, ptrs, &n, 1, out);
}

// ---- test hooks (not part of the reference-facing surface) ------------------------------------------------------------
// Evaluate the device build of the emulated libm: which = 0 asinf(a), 1 acosf(a), 2 atan2f(a, b), 3 atanf(a).
int urf_test_math(int device, int which, const float* a, const float* b, float* out, int n) {
  if (cudaSetDevice(device) != cudaSuccess) return URF_ERR_NO_DEVICE;
  float *da = nullptr, *db = nullptr, *dout = nullptr;
  if (cudaMalloc(&da, sizeof(float) * n) != cudaSuccess || cudaMalloc(&db, sizeof(float) * n) != cudaSuccess ||
      cudaMalloc(&dout, sizeof(float) * n) != cudaSuccess)
    return URF_ERR_NOMEM;
  cudaMemcpy(da, a, sizeof(float) * n, cudaMemcpyHostToDevice);
  cudaMemcpy(db, b ? b : a, sizeof(float) * n, cudaMemcpyHostToDevice);
  k_test_math<<<(n + 255) / 256, 256>>>(da, db, dout, n, which);
  cudaError_t e = cudaMemcpy(out, dout, sizeof(float) * n, cudaMemcpyDeviceToHost);
  cudaFree(da); cudaFree(db); cudaFree(dout);
  return e == cudaSuccess ? URF_OK : URF_ERR_CUDA;
}

// Copy a device-side intermediate of scan `b` of the last call into host memory (stage-level differential tests).
//   what: 0 alpha_v[f32,n]  1 mark[u8,n] (all detectors)  2 ringid[i16,n]  3 sect[i16,n]  4 az[f32,n]  5 d2[f32,n]
//         (4, 5: defined for ROI points only)  8 ScanTab (raw)
int urf_debug_fetch(urf_ctx* ctx, int b, int what, void* dst, size_t bytes) {
  if (!ctx || !dst || b < 0 || b >= ctx->last_B) return URF_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  const size_t off = (size_t)b * ctx->last_S;
  const void* src = nullptr;
  switch (what) {
    case 0: src = ctx->buf.alpha_v + off; break;
    case 1: src = ctx->buf.mark + off; break;
    case 2: src = ctx->buf.ringid + off; break;
    case 3: src = ctx->buf.sect + off; break;
    case 4: src = ctx->buf.az + off; break;
    case 5: src = ctx->buf.d2 + off; break;
    case 8: src = ctx->buf.tab + b; if (bytes > sizeof(ScanTab)) bytes = sizeof(ScanTab); break;
    default: return URF_ERR_INVALID;
  }
  CK(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
  return URF_OK;
}

size_t urf_debug_sizeof_tab(void) { return sizeof(ScanTab); }

}  // extern "C"
