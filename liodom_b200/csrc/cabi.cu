// C ABI of liodom_b200 (include/liodom_b200.h): context, device memory, host<->device
// staging and kernel orchestration. No CPU implementation of any stage lives here: if the
// CUDA device is missing the context cannot be created and every call fails.
#include "../../include/liodom_b200.h"
#include "common.cuh"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace liodom;

namespace liodom {
int launch_hash_begin_only(const DevBuffers& d, cudaStream_t s, int lane);
}

struct liodom_ctx {
  liodom_params params;
  int device = 0;
  int batch = 1;
  DevBuffers d{};        // with debug outputs
  DevBuffers dprod{};    // production view: debug pointers nulled
  cudaStream_t stream = nullptr, copy_stream = nullptr;
  // lane groups: a large batch is cut into `groups` ranges of lanes whose kernel chains run on their own streams,
  // so that the tail of one group's latency-bound kernels (k_associate, k_solve) overlaps another group's work
  static constexpr int kMaxGroups = 8;
  int groups = 1;
  bool groups_forced = false;   // LIODOM_LANE_GROUPS was set at creation
  cudaStream_t group_stream[kMaxGroups] = {};
  cudaEvent_t ev_fork = nullptr, ev_join[kMaxGroups] = {};
  std::vector<void*> allocs;
  std::string err;
  long long launches = 0;
  unsigned builds_since_clear = 0;
  // staging
  void* dev_in[2] = {nullptr, nullptr};
  size_t dev_in_bytes = 0;      // per buffer
  size_t dev_in_lane_bytes = 0;
  // Per scan in flight: B lane-indexed descriptors followed by the step's lane list (B ints; liodom_scan_lanes only),
  // staged in one pinned block and sent in one copy (see scan_batch_impl).  d_scan[0] == d.scan.
  ScanDesc* h_desc[2] = {nullptr, nullptr};   // pinned
  ScanDesc* d_scan[2] = {nullptr, nullptr};
  // A step that left lanes out (partial) reports n_edges = -1 for the lanes with stepped[buf][l] == 0.
  bool partial[2] = {false, false};
  std::vector<uint8_t> stepped[2];
  double* h_poses[2] = {nullptr, nullptr};    // pinned [B*16]
  int* h_nedges[2] = {nullptr, nullptr};      // pinned [B]
  cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
  bool in_flight[2] = {false, false};
  int cur = 0;                  // buffer of the last enqueued scan
  // scratch for single-lane API calls
  float4* stage_pts = nullptr;  // [max(Ecap, Mcap)]
  double* stage_cab = nullptr;  // [Ecap*9]
  double* stage_qt = nullptr;   // [16]
  SolveSummaryDev* stage_sum = nullptr;
  double* stage_pose = nullptr; // [12]
  ShardComm shard;              // point-sharded mode (liodom_shard_init); world == 1: off
  // optional per-stage device timing of liodom_scan_batch (bench roofline evidence)
  bool stage_timing = false;
  std::vector<cudaEvent_t> stage_events;  // LIODOM_NUM_STAGES + 1 events per timed call
  // LIODOM_TIMELINE=1: copy start/end and compute start/end of every liodom_scan_batch, printed at destroy
  bool timeline = false;
  std::vector<cudaEvent_t> tl_events;
};

// Record a stage boundary on the compute stream when stage timing is on.
static void stage_mark(liodom_ctx* c) {
  if (!c->stage_timing) return;
  cudaEvent_t e = nullptr;
  if (cudaEventCreate(&e) != cudaSuccess) return;
  cudaEventRecord(e, c->stream);
  c->stage_events.push_back(e);
}

static thread_local std::string g_create_err;

// Descriptor slots of one staging buffer: B descriptors, then room for a list of B lane indices.
static size_t desc_slots(int B) { return B + (sizeof(int32_t) * B + sizeof(ScanDesc) - 1) / sizeof(ScanDesc); }
static int32_t* lane_list(ScanDesc* descs, int B) { return reinterpret_cast<int32_t*>(descs + B); }

// Lane groups for a step of n lanes.  Measured at 128 lanes: 2 groups +4 %, 4 groups +0 %; at 32 lanes 2 groups -6 %.
static int default_lane_groups(int n) { return n >= 64 ? 2 : 1; }

static int fail(liodom_ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof(buf), fmt, ap); va_end(ap);
  if (c) c->err = buf; else g_create_err = buf;
  return code;
}

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) return fail(c, LIODOM_E_CUDA, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e_)); \
  } while (0)

template <typename T>
static cudaError_t dalloc(liodom_ctx* c, T** p, size_t count, bool zero = true) {
  void* q = nullptr;
  cudaError_t e = cudaMalloc(&q, count * sizeof(T) + 256);
  if (e != cudaSuccess) return e;
  c->allocs.push_back(q);
  if (zero) { e = cudaMemsetAsync(q, 0, count * sizeof(T) + 256, c->stream); if (e != cudaSuccess) return e; }
  *p = static_cast<T*>(q);
  return cudaSuccess;
}

static int ensure_dev_in(liodom_ctx* c, size_t lane_bytes) {
  if (lane_bytes <= c->dev_in_lane_bytes) return 0;
  for (int k = 0; k < 2; ++k) { if (c->dev_in[k]) cudaFree(c->dev_in[k]); c->dev_in[k] = nullptr; }
  const size_t lb = (lane_bytes + 255) / 256 * 256;
  for (int k = 0; k < 2; ++k) CK(cudaMalloc(&c->dev_in[k], lb * c->batch));
  c->dev_in_lane_bytes = lb; c->dev_in_bytes = lb * c->batch;
  return 0;
}

// The voxel hash tags entries with a 12-bit generation; clear the tables before it wraps.
static int hash_generation_guard(liodom_ctx* c, unsigned upcoming_builds) {
  c->builds_since_clear += upcoming_builds;
  if (c->builds_since_clear < 4000u) return 0;
  const DevBuffers& d = c->d;
  CK(cudaMemsetAsync(d.htab, 0, sizeof(HashEntry) * (size_t)d.p.Hcap * c->batch, c->stream));
  // reset every lane's generation counter and rebuild
  std::vector<WinState> ws(c->batch);
  CK(cudaMemcpyAsync(ws.data(), d.wstate, sizeof(WinState) * c->batch, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  for (auto& w : ws) { w.gen = 0; w.force_full = 1; w.built = 0; }
  CK(cudaMemcpyAsync(d.wstate, ws.data(), sizeof(WinState) * c->batch, cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  for (int l = 0; l < c->batch; ++l) c->launches += launch_hash_rebuild(d, c->stream, l);
  c->builds_since_clear = upcoming_builds + 1;
  return 0;
}

extern "C" {

void liodom_default_params(liodom_params* p) {
  p->min_range = 3.0; p->max_range = 75.0; p->lidar_type = 0; p->scan_lines = 64; p->scan_regions = 8;
  p->edges_per_region = 10; p->prev_frames = 5; p->filter_local_map = 0; p->mapping = 0;
  p->max_points = 262144; p->max_received_map = 0; p->use_imu = 0;
}

const char* liodom_last_error(const liodom_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }
int liodom_max_edges(const liodom_ctx* ctx) { return ctx->d.p.Ecap; }
void* liodom_stream(const liodom_ctx* ctx) { return ctx->stream; }
long long liodom_launch_count(const liodom_ctx* ctx) { return ctx->launches; }

int liodom_sync(liodom_ctx* c) {
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->copy_stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int liodom_ctx_create(const liodom_params* up, int batch, int device, liodom_ctx** out) {
  liodom_ctx* c = nullptr;
  if (!up || !out || batch < 1) return fail(nullptr, LIODOM_E_INVALID, "bad arguments");
  const liodom_params& P = *up;
  if (P.lidar_type != 0 && P.lidar_type != 1) return fail(nullptr, LIODOM_E_INVALID, "Incorrect Lidar type %d", P.lidar_type);
  if (P.lidar_type == 0 && P.scan_lines != 64 && P.scan_lines != 32 && P.scan_lines != 16)
    return fail(nullptr, LIODOM_E_INVALID, "Invalid scan lines: %d", P.scan_lines);
  if (P.scan_lines < 1 || P.scan_lines > kMaxLines) return fail(nullptr, LIODOM_E_INVALID, "scan_lines %d outside [1,%d]", P.scan_lines, kMaxLines);
  if (P.scan_regions < 1 || P.scan_regions > 256 || P.edges_per_region < 1 || P.edges_per_region > 255)
    return fail(nullptr, LIODOM_E_INVALID, "scan_regions/edges_per_region out of range");
  if (P.prev_frames < 1 || P.prev_frames + 1 > kMaxSlots) return fail(nullptr, LIODOM_E_INVALID, "prev_frames %d outside [1,%d]", P.prev_frames, kMaxSlots - 1);
  if (P.max_points < 1) return fail(nullptr, LIODOM_E_INVALID, "max_points must be positive");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || device < 0 || device >= ndev)
    return fail(nullptr, LIODOM_E_NODEVICE, "no usable CUDA device (count=%d, requested %d): liodom_b200 has no CPU fallback", ndev, device);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major < 10)
    return fail(nullptr, LIODOM_E_NODEVICE, "device %d is not sm_100-class (compute %d.%d)", device, prop.major, prop.minor);
  c = new liodom_ctx;
  c->params = P; c->device = device; c->batch = batch;
#define CKC(call)                                                                                  \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      fail(nullptr, LIODOM_E_CUDA, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e_)); \
      liodom_ctx_destroy(c);                                                                       \
      return LIODOM_E_CUDA;                                                                        \
    }                                                                                              \
  } while (0)
  CKC(cudaSetDevice(device));
  CKC(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  CKC(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  c->timeline = getenv("LIODOM_TIMELINE") != nullptr;
  {
    int g = default_lane_groups(batch);
    if (const char* e = getenv("LIODOM_LANE_GROUPS")) { g = atoi(e); c->groups_forced = true; }
    c->groups = std::max(1, std::min(std::min(g, batch), (int)liodom_ctx::kMaxGroups));
    CKC(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    for (int k = 0; k < c->groups && c->groups > 1; ++k) {
      CKC(cudaStreamCreateWithFlags(&c->group_stream[k], cudaStreamNonBlocking));
      CKC(cudaEventCreateWithFlags(&c->ev_join[k], cudaEventDisableTiming));
    }
  }
  DevBuffers& d = c->d;
  DevParams& p = d.p;
  p.min_range = P.min_range; p.max_range = P.max_range; p.lidar_type = P.lidar_type; p.scan_lines = P.scan_lines;
  p.scan_regions = P.scan_regions; p.edges_per_region = P.edges_per_region; p.prev_frames = P.prev_frames;
  p.filter_local_map = P.filter_local_map; p.mapping = P.mapping; p.use_imu = P.use_imu;
  p.batch = batch;
  p.Ncap = (P.max_points + kChunk - 1) / kChunk * kChunk;
  p.chunks = p.Ncap / kChunk;
  p.Ecap = P.scan_lines * P.scan_regions * (P.edges_per_region + 1);
  p.slots = P.prev_frames + 1;
  p.Wcap = p.slots * p.Ecap;
  // The per-cell point count shares a 32-bit word with the generation tag (kCntBits = 20 bits): keep the whole kNN
  // target below 2^20 points, then no cell can overflow its count even if every point fell into one voxel.
  const long long cnt_limit = (1ll << kCntBits) - 1;
  if ((long long)p.Wcap >= cnt_limit) {
    fail(nullptr, LIODOM_E_INVALID, "window of %d points (prev_frames+1 slabs x %d edges) exceeds the voxel-hash limit of %lld points", p.Wcap, p.Ecap, cnt_limit);
    liodom_ctx_destroy(c); return LIODOM_E_INVALID;
  }
  p.Rcap = P.mapping ? (P.max_received_map > 0 ? P.max_received_map : (int)std::min<long long>(1 << 20, cnt_limit - p.Wcap)) : 0;
  if ((long long)p.Wcap + p.Rcap > cnt_limit) {
    fail(nullptr, LIODOM_E_INVALID, "max_received_map %d + window %d exceed the voxel-hash limit of %lld points", p.Rcap, p.Wcap, cnt_limit);
    liodom_ctx_destroy(c); return LIODOM_E_INVALID;
  }
  p.Mcap = p.Wcap + p.Rcap;
  p.vg_blocks = (P.filter_local_map && !P.mapping) ? (p.Wcap + kVgTile - 1) / kVgTile : 0;
  int h = 1024; while (h < p.Mcap + p.Mcap / 8) h <<= 1;   // load factor <= 0.89 even if every point had its own voxel; typically < 0.2
  // The incremental hash (no mapping, no window filter) keeps emptied cells as tombstones until the next full build,
  // which it requests at half load: twice the slots.
  const bool incremental = !P.mapping && !P.filter_local_map;
  if (incremental) h <<= 1;
  p.Hcap = h;
  p.Pcap = incremental ? kPoolFactor * p.Mcap : p.Mcap;
  { int lc = 1024; while (lc < p.Mcap) lc <<= 1; p.LinCap = lc; }
  p.Bwords = h / 2;   // 16 filter bits per hash slot: a few % false positives (each costs one extra probe, never a wrong answer)
  if (extract_smem_needed(p) > (size_t)kMaxDynSmem) {
    fail(nullptr, LIODOM_E_INVALID, "scan_lines x scan_regions x edges_per_region needs %zu bytes of shared memory per CTA (limit %d)", extract_smem_needed(p), kMaxDynSmem);
    liodom_ctx_destroy(c); return LIODOM_E_INVALID;
  }
  CKC(configure_extract_kernels());   // per device: a second context on another GPU needs its own opt-in
  const size_t B = batch, L = P.scan_lines;
  CKC(dalloc(c, &d.scan, desc_slots(batch)));
  CKC(dalloc(c, &d.ring_id, B * p.Ncap, false));
  CKC(dalloc(c, &d.chunk_hist, B * p.chunks * L));
  CKC(dalloc(c, &d.chunk_base, B * p.chunks * L));
  CKC(dalloc(c, &d.chunk_amb, B * p.chunks));
  CKC(dalloc(c, &d.rings, B * p.Ncap, false));
  CKC(dalloc(c, &d.src_index, B * p.Ncap, false));
  CKC(dalloc(c, &d.ring_off, B * (L + 1)));
  CKC(dalloc(c, &d.keys, B * p.Ncap, false));
  CKC(dalloc(c, &d.pick_bits, B * 2 * ((size_t)(p.Ncap >> 5) + kMaxLines + 2)));
  CKC(dalloc(c, &d.slots, B * p.Ecap));
  CKC(dalloc(c, &d.slot_idx, B * p.Ecap));
  CKC(dalloc(c, &d.region_cnt, B * L * P.scan_regions));
  CKC(dalloc(c, &d.edges, B * p.Ecap));
  CKC(dalloc(c, &d.edge_ring, B * p.Ecap));
  CKC(dalloc(c, &d.edge_idx, B * p.Ecap));
  CKC(dalloc(c, &d.win, B * p.slots * p.Ecap));
  CKC(dalloc(c, &d.received, B * (size_t)(p.Rcap > 0 ? p.Rcap : 1)));
  CKC(dalloc(c, &d.wstate, B));
  CKC(dalloc(c, &d.ostate, B));
  CKC(dalloc(c, &d.sorted, B * p.Pcap));
  CKC(dalloc(c, &d.lin, B * p.LinCap));
  CKC(dalloc(c, &d.cap_end, B * p.Hcap));
  CKC(dalloc(c, &d.newcnt, B * p.Hcap));
  CKC(dalloc(c, &d.cell_base, B * p.Hcap));
  CKC(dalloc(c, &d.htab, B * p.Hcap));
  CKC(dalloc(c, &d.bloom, B * p.Bwords));
  CKC(dalloc(c, &d.owner_list, B * p.Mcap));
  CKC(dalloc(c, &d.pt_slot, B * p.Mcap));
  CKC(dalloc(c, &d.pt_rank, B * p.Mcap));
  CKC(dalloc(c, &d.perm, B * p.Ecap));
  CKC(dalloc(c, &d.knn_out, B * p.Ecap * 5));
  CKC(dalloc(c, &d.blocks, B * p.Ecap * 10));
  CKC(dalloc(c, &d.knn_idx, B * p.Ecap * 5));
  CKC(dalloc(c, &d.knn_d2, B * p.Ecap * 5));
  CKC(dalloc(c, &d.gate, B * p.Ecap));
  CKC(dalloc(c, &d.eig, B * p.Ecap * 3));
  CKC(dalloc(c, &d.q_world, B * p.Ecap));
  if (p.vg_blocks > 0) {   // filter_local_map: VoxelGrid of the window (voxelgrid.cu)
    CKC(dalloc(c, &d.filtered, B * p.Wcap, false));
    for (int k = 0; k < 2; ++k) { CKC(dalloc(c, &d.vg_key[k], B * p.Wcap, false)); CKC(dalloc(c, &d.vg_val[k], B * p.Wcap, false)); }
    CKC(dalloc(c, &d.vg_hist, B * 256 * p.vg_blocks));
    CKC(dalloc(c, &d.vg_heads, B * p.vg_blocks));
  }
  { unsigned char* q = nullptr; CKC(dalloc(c, &q, B * shard_ctrl_bytes())); d.shard_ctrl = q; }
  CKC(dalloc(c, &d.shard_acc, B * 32));
  CKC(dalloc(c, &d.diag, B));
  CKC(dalloc(c, &d.poses_out, B * 16));
  CKC(dalloc(c, &c->stage_pts, (size_t)(p.Mcap > p.Ecap ? p.Mcap : p.Ecap)));
  CKC(dalloc(c, &c->stage_cab, (size_t)p.Ecap * 9));
  CKC(dalloc(c, &c->stage_qt, 16));
  CKC(dalloc(c, &c->stage_sum, 1));
  CKC(dalloc(c, &c->stage_pose, 12));
  for (int k = 0; k < 2; ++k) {
    CKC(cudaMallocHost(&c->h_desc[k], sizeof(ScanDesc) * desc_slots(batch)));
    c->stepped[k].assign(B, 0);
    CKC(cudaMallocHost(&c->h_poses[k], sizeof(double) * 16 * B));
    CKC(cudaMallocHost(&c->h_nedges[k], sizeof(int) * B));
    CKC(cudaEventCreateWithFlags(&c->ev_copied[k], cudaEventDisableTiming));
    CKC(cudaEventCreateWithFlags(&c->ev_done[k], cudaEventDisableTiming));
  }
  c->d_scan[0] = d.scan;
  CKC(dalloc(c, &c->d_scan[1], desc_slots(batch)));
  c->dprod = c->d;
  c->dprod.gate = nullptr; c->dprod.knn_idx = nullptr; c->dprod.knn_d2 = nullptr; c->dprod.eig = nullptr;
  c->dprod.q_world = nullptr; c->dprod.src_index = nullptr;
  // initial state: identity poses, empty windows
  std::vector<OdomState> os(B);
  std::vector<WinState> ws(B);
  for (size_t l = 0; l < B; ++l) {
    std::memset(&os[l], 0, sizeof(OdomState)); std::memset(&ws[l], 0, sizeof(WinState));
    os[l].odom[0] = os[l].odom[5] = os[l].odom[10] = 1.0;
    os[l].prev[0] = os[l].prev[5] = os[l].prev[10] = 1.0;
    os[l].q[3] = 1.0;
    os[l].imu_q[3] = 1.0;
    os[l].l2b[0] = os[l].l2b[5] = os[l].l2b[10] = 1.0;
    ws[l].max_frames = P.prev_frames;
  }
  CKC(cudaMemcpyAsync(d.ostate, os.data(), sizeof(OdomState) * B, cudaMemcpyHostToDevice, c->stream));
  CKC(cudaMemcpyAsync(d.wstate, ws.data(), sizeof(WinState) * B, cudaMemcpyHostToDevice, c->stream));
  CKC(cudaStreamSynchronize(c->stream));
#undef CKC
  *out = c;
  return 0;
}

void liodom_ctx_destroy(liodom_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
  if (c->timeline && c->tl_events.size() >= 4) {
    for (size_t k = 0; k + 3 < c->tl_events.size(); k += 4) {
      float t[4];
      for (int j = 0; j < 4; ++j) cudaEventElapsedTime(&t[j], c->tl_events[0], c->tl_events[k + j]);
      fprintf(stderr, "[liodom timeline] step %zu: copy %.3f..%.3f  compute %.3f..%.3f ms\n", k / 4, t[0], t[1], t[2], t[3]);
    }
    for (cudaEvent_t e : c->tl_events) cudaEventDestroy(e);
  }
  for (void* p : c->allocs) cudaFree(p);
  for (int k = 0; k < 2; ++k) {
    if (c->dev_in[k]) cudaFree(c->dev_in[k]);
    if (c->h_desc[k]) cudaFreeHost(c->h_desc[k]);
    if (c->h_poses[k]) cudaFreeHost(c->h_poses[k]);
    if (c->h_nedges[k]) cudaFreeHost(c->h_nedges[k]);
    if (c->ev_copied[k]) cudaEventDestroy(c->ev_copied[k]);
    if (c->ev_done[k]) cudaEventDestroy(c->ev_done[k]);
  }
  shard_comm_destroy(&c->shard);
  for (int k = 0; k < liodom_ctx::kMaxGroups; ++k) {
    if (c->group_stream[k]) { cudaStreamSynchronize(c->group_stream[k]); cudaStreamDestroy(c->group_stream[k]); }
    if (c->ev_join[k]) cudaEventDestroy(c->ev_join[k]);
  }
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  for (cudaEvent_t e : c->stage_events) cudaEventDestroy(e);
  if (c->stream) cudaStreamDestroy(c->stream);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  delete c;
}

}  // extern "C"

// ---- helpers for the single-lane (facade / test) entry points ------------------------------
static int check_lane(liodom_ctx* c, int lane) {
  if (!c) return LIODOM_E_INVALID;
  if (lane < 0 || lane >= c->batch) return fail(c, LIODOM_E_INVALID, "lane %d outside [0,%d)", lane, c->batch);
  cudaError_t e = cudaSetDevice(c->device);
  if (e != cudaSuccess) return fail(c, LIODOM_E_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
  return 0;
}

// Where the four FLOAT32 fields of a point live (liodom_cloud_layout, or the fixed stride-only form).
struct Layout {
  int step = 16, row_step = 0, ox = 0, oy = 4, oz = 8, oi = 12, generic = 0;
};

static int layout_from_stride(liodom_ctx* c, int stride_bytes, Layout* L) {
  if (stride_bytes < 12 || (stride_bytes & 3)) return fail(c, LIODOM_E_INVALID, "bad stride_bytes %d", stride_bytes);
  *L = Layout{};
  L->step = stride_bytes;
  return 0;
}

// pcl::fromROSMsg (src/liodom_node.cc:43-44) copies each matched field byte for byte; it does not
// convert endianness, so big-endian messages are refused instead of decoded wrongly.
static int layout_from_user(liodom_ctx* c, const liodom_cloud_layout* u, int width, Layout* L) {
  if (!u) return fail(c, LIODOM_E_INVALID, "layout is NULL");
  if (u->is_bigendian) return fail(c, LIODOM_E_INVALID, "big-endian clouds are not supported (pcl::fromROSMsg copies bytes verbatim)");
  if (u->point_step < 12) return fail(c, LIODOM_E_INVALID, "point_step %d too small for x,y,z", u->point_step);
  const int offs[4] = {u->off_x, u->off_y, u->off_z, u->off_intensity};
  for (int k = 0; k < 4; ++k) {
    if (k == 3 && offs[k] < 0) continue;   // no intensity field: left 0
    if (offs[k] < 0 || offs[k] + 4 > u->point_step) return fail(c, LIODOM_E_INVALID, "field offset %d outside the %d-byte point", offs[k], u->point_step);
  }
  const long long packed_row = (long long)(width > 0 ? width : 0) * u->point_step;
  if (u->row_step != 0 && u->row_step < packed_row) return fail(c, LIODOM_E_INVALID, "row_step %d smaller than width * point_step", u->row_step);
  L->step = u->point_step;
  L->row_step = (u->row_step != 0 && u->row_step != packed_row) ? u->row_step : 0;
  L->ox = u->off_x; L->oy = u->off_y; L->oz = u->off_z; L->oi = u->off_intensity < 0 ? -1 : u->off_intensity;
  L->generic = 1;
  return 0;
}

static size_t scan_bytes(const Layout& L, int n, int width, int height) {
  if (L.generic && L.row_step && width > 0) return (size_t)(height > 0 ? height : (n + width - 1) / width) * L.row_step;
  return (size_t)n * L.step;
}

static void fill_desc(ScanDesc* sd, const void* pts, int n, const Layout& L, int width, int height) {
  sd->pts = pts; sd->n = n; sd->stride_bytes = L.step; sd->width = width > 0 ? width : 1; sd->height = height;
  sd->generic = L.generic; sd->row_step = L.row_step; sd->off_x = L.ox; sd->off_y = L.oy; sd->off_z = L.oz; sd->off_i = L.oi;
}

static int check_scan_shape(liodom_ctx* c, int lane, int n, const Layout& L, int width, int height) {
  if (n < 0 || n > c->d.p.Ncap) return fail(c, LIODOM_E_CAPACITY, "lane %d: %d points exceed max_points capacity %d", lane, n, c->d.p.Ncap);
  if (c->params.lidar_type == 1) {
    if (width <= 0 || height <= 0 || (long long)width * height != n) return fail(c, LIODOM_E_INVALID, "lane %d: organised cloud needs width*height == n", lane);
    if (height > c->params.scan_lines) return fail(c, LIODOM_E_INVALID, "cloud height %d exceeds scan_lines %d (the reference overruns its scans vector here)", height, c->params.scan_lines);
  }
  if (L.row_step && (width <= 0 || n % width != 0)) return fail(c, LIODOM_E_INVALID, "lane %d: padded rows need n to be a multiple of width", lane);
  return 0;
}

// Copy one host scan to the device staging area of `lane` (buffer 0) and publish its descriptor.
static int stage_scan(liodom_ctx* c, int lane, const void* pts, int n, const Layout& L, int width, int height) {
  int rc = check_scan_shape(c, lane, n, L, width, height); if (rc) return rc;
  const size_t bytes = scan_bytes(L, n, width, height);
  rc = ensure_dev_in(c, std::max((size_t)c->d.p.Ncap * 32, bytes));
  if (rc) return rc;
  char* dst = static_cast<char*>(c->dev_in[0]) + (size_t)lane * c->dev_in_lane_bytes;
  if (bytes > 0) CK(cudaMemcpyAsync(dst, pts, bytes, cudaMemcpyHostToDevice, c->stream));
  ScanDesc sd; fill_desc(&sd, dst, n, L, width, height);
  CK(cudaMemcpyAsync(c->d.scan + lane, &sd, sizeof(sd), cudaMemcpyHostToDevice, c->stream));
  return 0;
}

static int put_edges(liodom_ctx* c, int lane, const float* edges_xyzi, int n) {
  if (n < 0 || n > c->d.p.Ecap) return fail(c, LIODOM_E_CAPACITY, "%d edges exceed capacity %d", n, c->d.p.Ecap);
  if (n > 0) CK(cudaMemcpyAsync(c->d.edges + (size_t)lane * c->d.p.Ecap, edges_xyzi, (size_t)n * 16, cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemcpyAsync(&c->d.ostate[lane].n_edges, &n, sizeof(int), cudaMemcpyHostToDevice, c->stream));
  return 0;
}

static void pose12_from16(const double* p16, double* p12) { for (int k = 0; k < 12; ++k) p12[k] = p16[k]; }
static void pose16_from12(const double* p12, double* p16) { for (int k = 0; k < 12; ++k) p16[k] = p12[k]; p16[12] = p16[13] = p16[14] = 0.0; p16[15] = 1.0; }

static void copy_summary(const SolveSummaryDev& s, liodom_solve_summary* o) {
  o->iterations = s.iterations; o->successful_steps = s.successful_steps; o->termination = s.termination;
  o->num_residual_blocks = s.num_residual_blocks; o->cost_evals = s.cost_evals; o->jac_evals = s.jac_evals;
  o->initial_cost = s.initial_cost; o->final_cost = s.final_cost;
}

extern "C" {

int liodom_split(liodom_ctx* c, int lane, const void* pts, int n, int stride_bytes, int width, int height,
                 int32_t* ring_of_point, float* rings_xyzi, int32_t* ring_offsets, int32_t* src_index,
                 int* n_valid, int* n_ambiguous) {
  int rc = check_lane(c, lane); if (rc) return rc;
  Layout lay;
  rc = layout_from_stride(c, stride_bytes, &lay); if (rc) return rc;
  rc = stage_scan(c, lane, pts, n, lay, width, height); if (rc) return rc;
  const DevBuffers& d = c->d;
  c->launches += launch_split(d, c->stream, LaneRange{lane, 1});
  CK(cudaGetLastError());
  const int L = d.p.scan_lines;
  std::vector<int32_t> off(L + 1);
  std::vector<uint8_t> rid(n > 0 ? n : 1);
  OdomState os;
  CK(cudaMemcpyAsync(off.data(), d.ring_off + (size_t)lane * (L + 1), sizeof(int32_t) * (L + 1), cudaMemcpyDeviceToHost, c->stream));
  if (n > 0) CK(cudaMemcpyAsync(rid.data(), d.ring_id + (size_t)lane * d.p.Ncap, n, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(&os, d.ostate + lane, sizeof(os), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  const int nv = off[L];
  if (rings_xyzi && nv > 0) CK(cudaMemcpy(rings_xyzi, d.rings + (size_t)lane * d.p.Ncap, (size_t)nv * 16, cudaMemcpyDeviceToHost));
  if (src_index && nv > 0) CK(cudaMemcpy(src_index, d.src_index + (size_t)lane * d.p.Ncap, (size_t)nv * 4, cudaMemcpyDeviceToHost));
  if (ring_offsets) std::memcpy(ring_offsets, off.data(), sizeof(int32_t) * (L + 1));
  if (ring_of_point) for (int i = 0; i < n; ++i) ring_of_point[i] = rid[i] == 255 ? -1 : (int32_t)rid[i];
  if (n_valid) *n_valid = nv;
  if (n_ambiguous) *n_ambiguous = os.n_ambiguous;
  return 0;
}

static int extract_impl(liodom_ctx* c, int lane, const void* pts, int n, const Layout& lay, int width, int height,
                        float* edges_xyzi, int* n_edges, int32_t* edge_ring, int32_t* edge_idx, double* keys);

int liodom_extract(liodom_ctx* c, int lane, const void* pts, int n, int stride_bytes, int width, int height,
                   float* edges_xyzi, int* n_edges, int32_t* edge_ring, int32_t* edge_idx, double* keys) {
  int rc = check_lane(c, lane); if (rc) return rc;
  Layout lay;
  rc = layout_from_stride(c, stride_bytes, &lay); if (rc) return rc;
  return extract_impl(c, lane, pts, n, lay, width, height, edges_xyzi, n_edges, edge_ring, edge_idx, keys);
}

int liodom_extract_layout(liodom_ctx* c, int lane, const void* data, int n, const liodom_cloud_layout* layout, int width, int height,
                          float* edges_xyzi, int* n_edges, int32_t* edge_ring, int32_t* edge_idx) {
  int rc = check_lane(c, lane); if (rc) return rc;
  Layout lay;
  rc = layout_from_user(c, layout, width, &lay); if (rc) return rc;
  return extract_impl(c, lane, data, n, lay, width, height, edges_xyzi, n_edges, edge_ring, edge_idx, nullptr);
}

static int extract_impl(liodom_ctx* c, int lane, const void* pts, int n, const Layout& lay, int width, int height,
                        float* edges_xyzi, int* n_edges, int32_t* edge_ring, int32_t* edge_idx, double* keys) {
  int rc = stage_scan(c, lane, pts, n, lay, width, height); if (rc) return rc;
  const DevBuffers& d = c->dprod;
  if (keys) CK(cudaMemsetAsync(d.keys + (size_t)lane * d.p.Ncap, 0xff, sizeof(double) * d.p.Ncap, c->stream));  // NaN
  c->launches += launch_split(d, c->stream, LaneRange{lane, 1});
  c->launches += launch_extract(d, c->stream, LaneRange{lane, 1}, keys != nullptr);
  CK(cudaGetLastError());
  OdomState os;
  CK(cudaMemcpyAsync(&os, d.ostate + lane, sizeof(os), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  const int E = os.n_edges;
  if (n_edges) *n_edges = E;
  if (E > 0) {
    if (edges_xyzi) CK(cudaMemcpy(edges_xyzi, d.edges + (size_t)lane * d.p.Ecap, (size_t)E * 16, cudaMemcpyDeviceToHost));
    if (edge_ring) CK(cudaMemcpy(edge_ring, d.edge_ring + (size_t)lane * d.p.Ecap, (size_t)E * 4, cudaMemcpyDeviceToHost));
    if (edge_idx) CK(cudaMemcpy(edge_idx, d.edge_idx + (size_t)lane * d.p.Ecap, (size_t)E * 4, cudaMemcpyDeviceToHost));
  }
  if (keys && os.n_valid > 0) CK(cudaMemcpy(keys, d.keys + (size_t)lane * d.p.Ncap, sizeof(double) * os.n_valid, cudaMemcpyDeviceToHost));
  return 0;
}

int liodom_lmap_add(liodom_ctx* c, int lane, const float* xyzi, int n) {
  int rc = check_lane(c, lane); if (rc) return rc;
  if (n < 0 || n > c->d.p.Ecap) return fail(c, LIODOM_E_CAPACITY, "frame of %d points exceeds the slab capacity %d", n, c->d.p.Ecap);
  rc = hash_generation_guard(c, 1); if (rc) return rc;
  if (n > 0) CK(cudaMemcpyAsync(c->stage_pts, xyzi, (size_t)n * 16, cudaMemcpyHostToDevice, c->stream));
  c->launches += launch_lmap_add(c->d, c->stream, lane, c->stage_pts, n);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int liodom_lmap_get(liodom_ctx* c, int lane, float* xyzi, int cap, int* n_points, int* n_frames) {
  int rc = check_lane(c, lane); if (rc) return rc;
  WinState ws;
  CK(cudaMemcpyAsync(&ws, c->d.wstate + lane, sizeof(ws), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (n_points) *n_points = ws.total;
  if (n_frames) *n_frames = ws.nframes;
  if (xyzi && ws.total > 0) {
    if (cap < ws.total) return fail(c, LIODOM_E_CAPACITY, "output capacity %d < window size %d", cap, ws.total);
    c->launches += launch_lmap_gather(c->d, c->stream, lane, c->stage_pts);
    CK(cudaMemcpyAsync(xyzi, c->stage_pts, (size_t)ws.total * 16, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
  }
  return 0;
}

int liodom_lmap_set_max_frames(liodom_ctx* c, int lane, int max_frames) {
  int rc = check_lane(c, lane); if (rc) return rc;
  if (max_frames < 0 || max_frames + 1 > c->d.p.slots)
    return fail(c, LIODOM_E_CAPACITY, "max_frames %d needs %d slabs, context was created with %d (prev_frames)", max_frames, max_frames + 1, c->d.p.slots);
  CK(cudaMemcpyAsync(&c->d.wstate[lane].max_frames, &max_frames, sizeof(int), cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int liodom_lmap_clear(liodom_ctx* c, int lane) {
  int rc = check_lane(c, lane); if (rc) return rc;
  WinState ws;
  CK(cudaMemcpyAsync(&ws, c->d.wstate + lane, sizeof(ws), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  const unsigned gen = ws.gen; const int mf = ws.max_frames, nr = ws.n_received;
  std::memset(&ws, 0, sizeof(ws));
  ws.gen = gen; ws.max_frames = mf; ws.n_received = nr; ws.force_full = 1;
  CK(cudaMemcpyAsync(c->d.wstate + lane, &ws, sizeof(ws), cudaMemcpyHostToDevice, c->stream));
  rc = hash_generation_guard(c, 1); if (rc) return rc;
  c->launches += launch_hash_rebuild(c->d, c->stream, lane);
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int liodom_set_received_map(liodom_ctx* c, int lane, const float* xyzi, int n) {
  int rc = check_lane(c, lane); if (rc) return rc;
  if (!c->params.mapping) return fail(c, LIODOM_E_INVALID, "context was created with mapping=0");
  if (n < 0 || n > c->d.p.Rcap) return fail(c, LIODOM_E_CAPACITY, "received map of %d points exceeds max_received_map %d", n, c->d.p.Rcap);
  if (n > 0) CK(cudaMemcpyAsync(c->d.received + (size_t)lane * c->d.p.Rcap, xyzi, (size_t)n * 16, cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemcpyAsync(&c->d.wstate[lane].n_received, &n, sizeof(int), cudaMemcpyHostToDevice, c->stream));
  rc = hash_generation_guard(c, 1); if (rc) return rc;
  c->launches += launch_hash_rebuild(c->d, c->stream, lane);
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

// Device-side variant of liodom_set_received_map: the caller (e.g. liodom_map_get_local_device) writes
// the cloud straight into the lane's received-map buffer, then commits its size.
int liodom_received_map_buffer(liodom_ctx* c, int lane, void** dev_xyzi, int* cap) {
  int rc = check_lane(c, lane); if (rc) return rc;
  if (!c->params.mapping) return fail(c, LIODOM_E_INVALID, "context was created with mapping=0");
  // The producer writes on ITS stream: scans still in flight here (their hash build reads this buffer) must finish first.
  rc = liodom_sync(c); if (rc) return rc;
  if (dev_xyzi) *dev_xyzi = c->d.received + (size_t)lane * c->d.p.Rcap;
  if (cap) *cap = c->d.p.Rcap;
  return 0;
}

int liodom_commit_received_map(liodom_ctx* c, int lane, int n) {
  int rc = check_lane(c, lane); if (rc) return rc;
  if (!c->params.mapping) return fail(c, LIODOM_E_INVALID, "context was created with mapping=0");
  if (n < 0 || n > c->d.p.Rcap) return fail(c, LIODOM_E_CAPACITY, "received map of %d points exceeds max_received_map %d", n, c->d.p.Rcap);
  CK(cudaMemcpyAsync(&c->d.wstate[lane].n_received, &n, sizeof(int), cudaMemcpyHostToDevice, c->stream));
  rc = hash_generation_guard(c, 1); if (rc) return rc;
  c->launches += launch_hash_rebuild(c->d, c->stream, lane);
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int liodom_odom_reset(liodom_ctx* c, int lane) {
  int rc = check_lane(c, lane); if (rc) return rc;
  OdomState os; std::memset(&os, 0, sizeof(os));
  os.odom[0] = os.odom[5] = os.odom[10] = 1.0; os.prev[0] = os.prev[5] = os.prev[10] = 1.0; os.q[3] = 1.0;
  os.imu_q[3] = 1.0; os.l2b[0] = os.l2b[5] = os.l2b[10] = 1.0;
  CK(cudaMemcpyAsync(c->d.ostate + lane, &os, sizeof(os), cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return liodom_lmap_clear(c, lane);
}

int liodom_odom_set_pose(liodom_ctx* c, int lane, const double* odom16, const double* prev16) {
  int rc = check_lane(c, lane); if (rc) return rc;
  OdomState os;
  CK(cudaMemcpyAsync(&os, c->d.ostate + lane, sizeof(os), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (odom16) pose12_from16(odom16, os.odom);
  if (prev16) pose12_from16(prev16, os.prev);
  os.init = 1;
  CK(cudaMemcpyAsync(c->d.ostate + lane, &os, sizeof(os), cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int liodom_odom_set_imu(liodom_ctx* c, int lane, const double* q_xyzw) {
  int rc = check_lane(c, lane); if (rc) return rc;
  if (!q_xyzw) return fail(c, LIODOM_E_INVALID, "q_xyzw is NULL");
  CK(cudaMemcpyAsync(c->d.ostate[lane].imu_q, q_xyzw, sizeof(double) * 4, cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));   // the caller's buffer may be a temporary
  return 0;
}

int liodom_odom_set_laser_to_base(liodom_ctx* c, int lane, const double* T16) {
  int rc = check_lane(c, lane); if (rc) return rc;
  if (!T16) return fail(c, LIODOM_E_INVALID, "T16 is NULL");
  CK(cudaMemcpyAsync(c->d.ostate[lane].l2b, T16, sizeof(double) * 12, cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int liodom_odom_get_pose(liodom_ctx* c, int lane, double* odom16, double* prev16) {
  int rc = check_lane(c, lane); if (rc) return rc;
  OdomState os;
  CK(cudaMemcpyAsync(&os, c->d.ostate + lane, sizeof(os), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (odom16) pose16_from12(os.odom, odom16);
  if (prev16) pose16_from12(os.prev, prev16);
  return 0;
}

int liodom_associate(liodom_ctx* c, int lane, const float* edges_xyzi, int n_edges, const double* pose16,
                     int32_t* knn_idx, float* knn_d2, uint8_t* gate, double* eig, float* q_world, int* n_map) {
  int rc = check_lane(c, lane); if (rc) return rc;
  rc = put_edges(c, lane, edges_xyzi, n_edges); if (rc) return rc;
  const DevBuffers& d = c->d;
  const double* pose_dev = nullptr;
  if (pose16) { CK(cudaMemcpyAsync(c->stage_pose, pose16, sizeof(double) * 12, cudaMemcpyHostToDevice, c->stream)); pose_dev = c->stage_pose; }
  c->launches += launch_associate(d, c->stream, LaneRange{lane, 1}, 0, true, pose_dev);
  CK(cudaGetLastError());
  const size_t o = (size_t)lane * d.p.Ecap, E = n_edges;
  if (E > 0) {
    if (knn_idx) CK(cudaMemcpyAsync(knn_idx, d.knn_idx + o * 5, E * 20, cudaMemcpyDeviceToHost, c->stream));
    if (knn_d2) CK(cudaMemcpyAsync(knn_d2, d.knn_d2 + o * 5, E * 20, cudaMemcpyDeviceToHost, c->stream));
    if (gate) CK(cudaMemcpyAsync(gate, d.gate + o, E, cudaMemcpyDeviceToHost, c->stream));
    if (eig) CK(cudaMemcpyAsync(eig, d.eig + o * 3, E * 24, cudaMemcpyDeviceToHost, c->stream));
    if (q_world) CK(cudaMemcpyAsync(q_world, d.q_world + o, E * 16, cudaMemcpyDeviceToHost, c->stream));
  }
  WinState ws;
  CK(cudaMemcpyAsync(&ws, d.wstate + lane, sizeof(ws), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (n_map) *n_map = ws.hash_points;
  return 0;
}

int liodom_solve(liodom_ctx* c, int lane, const double* cab, int n, double* q4, double* t3, liodom_solve_summary* summary) {
  int rc = check_lane(c, lane); if (rc) return rc;
  if (n < 0 || n > c->d.p.Ecap) return fail(c, LIODOM_E_CAPACITY, "%d residual blocks exceed capacity %d", n, c->d.p.Ecap);
  double qt[7] = {q4[0], q4[1], q4[2], q4[3], t3[0], t3[1], t3[2]};
  if (n > 0) CK(cudaMemcpyAsync(c->stage_cab, cab, sizeof(double) * 9 * n, cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemcpyAsync(c->stage_qt, qt, sizeof(qt), cudaMemcpyHostToDevice, c->stream));
  c->launches += launch_solve_blocks(c->d, c->stream, lane, c->stage_cab, n, c->stage_qt, c->stage_sum);
  CK(cudaGetLastError());
  SolveSummaryDev s;
  CK(cudaMemcpyAsync(qt, c->stage_qt, sizeof(qt), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(&s, c->stage_sum, sizeof(s), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  for (int k = 0; k < 4; ++k) q4[k] = qt[k];
  for (int k = 0; k < 3; ++k) t3[k] = qt[4 + k];
  if (summary) copy_summary(s, summary);
  return 0;
}

static int enqueue_register(liodom_ctx* c, const DevBuffers& d, LaneRange lr) {
  int k = 0;
  k += launch_predict(d, c->stream, lr);
  for (int it = 0; it < 2; ++it) {  // src/laser_odometry.cc:198
    k += launch_associate(d, c->stream, lr, it, false, nullptr);
    stage_mark(c);
    k += launch_solve(d, c->stream, lr, it);
    stage_mark(c);
  }
  k += launch_window_update(d, c->stream, lr);
  stage_mark(c);
  return k;
}

// Point-sharded scan (one lane): ring-sharded extraction + all-gather of the edge slots, replicated
// prediction / ordering / window, edge-sharded association and solve with a 29-double all-reduce per
// LM evaluation.
static int enqueue_scan_sharded(liodom_ctx* c, const DevBuffers& d, int* launches) {
  const ShardComm* sc = &c->shard;
  const LaneRange lr{0, 1};
  const int L = d.p.scan_lines, per = L / sc->world;
  const size_t slots_per_rank = (size_t)per * d.p.scan_regions * (d.p.edges_per_region + 1);
  int k = 0, nrc = 0;
  stage_mark(c);
  k += launch_split(d, c->stream, lr);
  stage_mark(c);
  k += launch_extract_rings(d, c->stream, lr, sc->rank * per, per);
  nrc |= shard_group_start();
  nrc |= shard_allgather_bytes(sc, d.slots, slots_per_rank * sizeof(float4), c->stream);
  nrc |= shard_allgather_bytes(sc, d.slot_idx, slots_per_rank * sizeof(int), c->stream);
  nrc |= shard_allgather_bytes(sc, d.region_cnt, (size_t)per * d.p.scan_regions * sizeof(int), c->stream);
  nrc |= shard_group_end();
  k += launch_compact(d, c->stream, lr);
  stage_mark(c);
  k += launch_predict(d, c->stream, lr);
  for (int it = 0; it < 2; ++it) {
    k += launch_associate_shard(d, c->stream, 0, it, sc->rank, sc->world);
    stage_mark(c);
    k += launch_solve_shard(d, c->stream, 0, it, sc, &nrc);
    stage_mark(c);
  }
  k += launch_window_update(d, c->stream, lr);
  stage_mark(c);
  *launches = k;
  if (nrc != 0) return fail(c, LIODOM_E_CUDA, "NCCL call failed in the point-sharded scan: %s", shard_error_string(nrc));
  return 0;
}

int liodom_shard_unique_id(char id_out[128]) {
  const int rc = shard_unique_id(id_out);
  if (rc != 0) return fail(nullptr, LIODOM_E_INVALID, "ncclGetUniqueId: %s", shard_error_string(rc));
  return 0;
}

int liodom_shard_init(liodom_ctx* c, int rank, int world, const char id[128]) {
  if (!c || !id) return LIODOM_E_INVALID;
  CK(cudaSetDevice(c->device));
  if (c->batch != 1) return fail(c, LIODOM_E_INVALID, "point-sharded mode needs a batch-1 context");
  if (world < 1 || rank < 0 || rank >= world) return fail(c, LIODOM_E_INVALID, "bad rank/world (%d/%d)", rank, world);
  if (c->params.scan_lines % world != 0) return fail(c, LIODOM_E_INVALID, "scan_lines %d is not a multiple of the world size %d", c->params.scan_lines, world);
  shard_comm_destroy(&c->shard);
  if (world == 1) return 0;
  const int rc = shard_comm_init(&c->shard, rank, world, id);
  if (rc != 0) return fail(c, LIODOM_E_CUDA, "ncclCommInitRank: %s", shard_error_string(rc));
  return 0;
}

int liodom_register(liodom_ctx* c, int lane, const float* edges_xyzi, int n_edges, double* pose16_out, liodom_frame_diag* diag) {
  int rc = check_lane(c, lane); if (rc) return rc;
  rc = hash_generation_guard(c, 1); if (rc) return rc;
  rc = put_edges(c, lane, edges_xyzi, n_edges); if (rc) return rc;
  const DevBuffers& d = c->dprod;
  const bool st = c->stage_timing;  // stage timing covers liodom_scan_batch only
  c->stage_timing = false;
  c->launches += enqueue_register(c, d, LaneRange{lane, 1});
  c->stage_timing = st;
  CK(cudaGetLastError());
  double pose[16]; FrameDiagDev dg;
  CK(cudaMemcpyAsync(pose, d.poses_out + (size_t)lane * 16, sizeof(pose), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(&dg, d.diag + lane, sizeof(dg), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (pose16_out) std::memcpy(pose16_out, pose, sizeof(pose));
  if (diag) {
    diag->n_edges = n_edges;
    for (int k = 0; k < 2; ++k) { diag->n_map[k] = dg.n_map[k]; diag->n_matches[k] = dg.n_matches[k]; copy_summary(dg.solve[k], &diag->solve[k]); }
    std::memcpy(diag->pred_pose, dg.pred_pose, sizeof(dg.pred_pose));
  }
  return 0;
}

// ---- whole hot path, batched --------------------------------------------------------------
// lanes == nullptr: every lane, position l = lane l (liodom_scan_batch).  Otherwise position i steps lane lanes[i].
static int scan_batch_impl(liodom_ctx* c, const int32_t* lanes, int n_lanes, const void* const* pts, const int* n, const Layout& lay,
                           int width, int height, int on_device);

int liodom_scan_batch(liodom_ctx* c, const void* const* pts, const int* n, int stride_bytes, int width, int height, int on_device) {
  if (!c) return LIODOM_E_INVALID;
  Layout lay;
  int rc = layout_from_stride(c, stride_bytes, &lay); if (rc) return rc;
  return scan_batch_impl(c, nullptr, c->batch, pts, n, lay, width, height, on_device);
}

int liodom_scan_batch_layout(liodom_ctx* c, const void* const* data, const int* n, const liodom_cloud_layout* layout, int width, int height, int on_device) {
  if (!c) return LIODOM_E_INVALID;
  Layout lay;
  int rc = layout_from_user(c, layout, width, &lay); if (rc) return rc;
  return scan_batch_impl(c, nullptr, c->batch, data, n, lay, width, height, on_device);
}

// A lane list from the caller: in range, no duplicates, not on a point-sharded context.
static int check_lane_list(liodom_ctx* c, const int32_t* lanes, int n_lanes, const void* const* pts, const int* n) {
  if (c->shard.world > 1) return fail(c, LIODOM_E_INVALID, "a point-sharded context steps its one lane with liodom_scan_batch");
  if (n_lanes < 0 || n_lanes > c->batch) return fail(c, LIODOM_E_INVALID, "n_lanes %d outside [0,%d]", n_lanes, c->batch);
  if (n_lanes > 0 && (!lanes || !pts || !n)) return fail(c, LIODOM_E_INVALID, "lanes, pts and n must not be NULL");
  std::vector<uint8_t> seen(c->batch, 0);
  for (int i = 0; i < n_lanes; ++i) {
    const int l = lanes[i];
    if (l < 0 || l >= c->batch) return fail(c, LIODOM_E_INVALID, "lanes[%d] = %d outside [0,%d)", i, l, c->batch);
    if (seen[l]) return fail(c, LIODOM_E_INVALID, "lane %d listed twice", l);
    seen[l] = 1;
  }
  return 0;
}

int liodom_scan_lanes(liodom_ctx* c, const int32_t* lanes, int n_lanes, const void* const* pts, const int* n, int stride_bytes,
                      int width, int height, int on_device) {
  if (!c) return LIODOM_E_INVALID;
  int rc = check_lane_list(c, lanes, n_lanes, pts, n); if (rc) return rc;
  Layout lay;
  rc = layout_from_stride(c, stride_bytes, &lay); if (rc) return rc;
  return scan_batch_impl(c, lanes, n_lanes, pts, n, lay, width, height, on_device);
}

int liodom_scan_lanes_layout(liodom_ctx* c, const int32_t* lanes, int n_lanes, const void* const* data, const int* n,
                             const liodom_cloud_layout* layout, int width, int height, int on_device) {
  if (!c) return LIODOM_E_INVALID;
  int rc = check_lane_list(c, lanes, n_lanes, data, n); if (rc) return rc;
  Layout lay;
  rc = layout_from_user(c, layout, width, &lay); if (rc) return rc;
  return scan_batch_impl(c, lanes, n_lanes, data, n, lay, width, height, on_device);
}

static int scan_batch_impl(liodom_ctx* c, const int32_t* lanes, int n_lanes, const void* const* pts, const int* n, const Layout& lay,
                           int width, int height, int on_device) {
  CK(cudaSetDevice(c->device));
  if (n_lanes == 0) return 0;
  const int B = c->batch;
  auto lane_of = [&](int i) { return lanes ? (int)lanes[i] : i; };
  int rc;
  for (int i = 0; i < n_lanes; ++i) { rc = check_scan_shape(c, lane_of(i), n[i], lay, width, height); if (rc) return rc; }
  rc = hash_generation_guard(c, 1); if (rc) return rc;
  const int buf = c->cur ^ 1;
  if (c->in_flight[buf]) { CK(cudaEventSynchronize(c->ev_done[buf])); c->in_flight[buf] = false; }
  ScanDesc* hd = c->h_desc[buf];
  // Descriptors stay lane-indexed (only the listed lanes' are rewritten); the list rides in the same copy.
  if (lanes) std::memcpy(lane_list(hd, B), lanes, sizeof(int32_t) * n_lanes);
  const size_t desc_bytes = sizeof(ScanDesc) * B + (lanes ? sizeof(int32_t) * n_lanes : 0);
  if (!on_device) {
    size_t max_bytes = (size_t)c->d.p.Ncap * 32;
    for (int i = 0; i < n_lanes; ++i) max_bytes = std::max(max_bytes, scan_bytes(lay, n[i], width, height));
    rc = ensure_dev_in(c, max_bytes); if (rc) return rc;
    // Host scans laid out back to back in list order (a batching front-end would do that) go over PCIe as ONE copy
    // into a packed staging area; otherwise one copy per list position into fixed-pitch slots.
    bool packed = n_lanes > 1 && (lay.step & 3) == 0 && !lay.row_step;   // 4-byte aligned records (16-byte xyzi, 32-byte PCL, 12-byte xyz)
    size_t total = 0;
    for (int i = 0; i < n_lanes && packed; ++i) {
      if (static_cast<const char*>(pts[i]) != static_cast<const char*>(pts[0]) + total) packed = false;
      total += (size_t)n[i] * lay.step;
    }
    packed = packed && total <= c->dev_in_bytes;
    size_t off = 0;
    for (int i = 0; i < n_lanes; ++i) {
      char* dst = packed ? static_cast<char*>(c->dev_in[buf]) + off : static_cast<char*>(c->dev_in[buf]) + (size_t)i * c->dev_in_lane_bytes;
      fill_desc(&hd[lane_of(i)], dst, n[i], lay, width, height);
      off += (size_t)n[i] * lay.step;
    }
    // The descriptors go FIRST and on the copy stream: a small H2D copy issued on the compute stream would
    // queue behind the next scan's bulk copy on the same copy engine and stall this scan's kernels for
    // the whole transfer (measured: 6.6 ms instead of 2.7 ms of compute per second step at 128 lanes).
    CK(cudaMemcpyAsync(c->d_scan[buf], hd, desc_bytes, cudaMemcpyHostToDevice, c->copy_stream));
    if (c->timeline) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, c->copy_stream); c->tl_events.push_back(e); }
    if (packed) {
      if (total > 0) CK(cudaMemcpyAsync(c->dev_in[buf], pts[0], total, cudaMemcpyHostToDevice, c->copy_stream));
    } else {
      for (int i = 0; i < n_lanes; ++i) {
        const size_t bytes = scan_bytes(lay, n[i], width, height);
        if (bytes > 0) CK(cudaMemcpyAsync(const_cast<void*>(hd[lane_of(i)].pts), pts[i], bytes, cudaMemcpyHostToDevice, c->copy_stream));
      }
    }
    if (c->timeline) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, c->copy_stream); c->tl_events.push_back(e); }
    CK(cudaEventRecord(c->ev_copied[buf], c->copy_stream));
    CK(cudaStreamWaitEvent(c->stream, c->ev_copied[buf], 0));
    if (c->timeline) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, c->stream); c->tl_events.push_back(e); }
  } else {
    for (int i = 0; i < n_lanes; ++i) fill_desc(&hd[lane_of(i)], pts[i], n[i], lay, width, height);
    CK(cudaMemcpyAsync(c->d_scan[buf], hd, desc_bytes, cudaMemcpyHostToDevice, c->stream));
  }
  DevBuffers d = c->dprod;
  d.scan = c->d_scan[buf];
  d.lanes = lanes ? lane_list(c->d_scan[buf], B) : nullptr;
  const LaneRange lr{0, n_lanes};
  // the lane groups a context of n_lanes lanes would use, at most the streams this one has
  const int G = std::min(std::min(c->groups, n_lanes), c->groups_forced ? c->groups : default_lane_groups(n_lanes));
  int k = 0;
  if (c->shard.world > 1) {
    rc = enqueue_scan_sharded(c, d, &k);
    if (rc) return rc;
  } else if (G > 1 && !c->stage_timing) {
    // fork: every group's chain waits for the descriptors (and the H2D copy) on the main stream
    CK(cudaEventRecord(c->ev_fork, c->stream));
    for (int g = 0; g < G; ++g) CK(cudaStreamWaitEvent(c->group_stream[g], c->ev_fork, 0));
    for (int st = 0; st < 7; ++st)
      for (int g = 0; g < G; ++g) {
        const int l0 = (int)((long long)n_lanes * g / G), l1 = (int)((long long)n_lanes * (g + 1) / G);
        const LaneRange gr{l0, l1 - l0};
        cudaStream_t s = c->group_stream[g];
        {
          switch (st) {
            case 0: k += launch_split(d, s, gr); break;
            case 1: k += launch_extract(d, s, gr, false); break;
            case 2: k += launch_predict(d, s, gr); k += launch_associate(d, s, gr, 0, false, nullptr); break;
            case 3: k += launch_solve(d, s, gr, 0); break;
            case 4: k += launch_associate(d, s, gr, 1, false, nullptr); break;
            case 5: k += launch_solve(d, s, gr, 1); break;
            default: k += launch_window_update(d, s, gr); break;
          }
        }
      }
    for (int g = 0; g < G; ++g) {   // join
      CK(cudaEventRecord(c->ev_join[g], c->group_stream[g]));
      CK(cudaStreamWaitEvent(c->stream, c->ev_join[g], 0));
    }
  } else {
    stage_mark(c);
    k += launch_split(d, c->stream, lr);
    stage_mark(c);
    k += launch_extract(d, c->stream, lr, false);
    stage_mark(c);
    k += enqueue_register(c, d, lr);
  }
  c->launches += k;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(c->h_poses[buf], d.poses_out, sizeof(double) * 16 * B, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpy2DAsync(c->h_nedges[buf], sizeof(int), &d.ostate[0].n_edges, sizeof(OdomState), sizeof(int), B, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaEventRecord(c->ev_done[buf], c->stream));
  if (c->timeline && !on_device) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, c->stream); c->tl_events.push_back(e); }
  c->in_flight[buf] = true;
  c->cur = buf;
  c->partial[buf] = n_lanes < B;
  if (c->partial[buf]) {
    std::fill(c->stepped[buf].begin(), c->stepped[buf].end(), 0);
    for (int i = 0; i < n_lanes; ++i) c->stepped[buf][lanes[i]] = 1;
  }
  return 0;
}

int liodom_stage_timing(liodom_ctx* c, int enable) {
  if (!c) return LIODOM_E_INVALID;
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  for (cudaEvent_t e : c->stage_events) cudaEventDestroy(e);
  c->stage_events.clear();
  c->stage_timing = enable != 0;
  return 0;
}

int liodom_stage_times(liodom_ctx* c, double* ms_out, int* n_calls) {
  if (!c || !ms_out) return LIODOM_E_INVALID;
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  const size_t per = LIODOM_NUM_STAGES + 1;
  const size_t calls = c->stage_events.size() / per;
  for (int s = 0; s < LIODOM_NUM_STAGES; ++s) ms_out[s] = 0.0;
  for (size_t k = 0; k < calls; ++k)
    for (int s = 0; s < LIODOM_NUM_STAGES; ++s) {
      float ms = 0.f;
      CK(cudaEventElapsedTime(&ms, c->stage_events[k * per + s], c->stage_events[k * per + s + 1]));
      ms_out[s] += ms;
    }
  if (n_calls) *n_calls = (int)calls;
  return 0;
}

int liodom_scan_results_of(liodom_ctx* c, int age, double* poses16_out, int* n_edges_out) {
  if (!c) return LIODOM_E_INVALID;
  if (age != 0 && age != 1) return fail(c, LIODOM_E_INVALID, "age must be 0 (last enqueued scan) or 1 (the one before)");
  CK(cudaSetDevice(c->device));
  const int buf = c->cur ^ age;
  if (c->in_flight[buf]) { CK(cudaEventSynchronize(c->ev_done[buf])); c->in_flight[buf] = false; }
  if (poses16_out) std::memcpy(poses16_out, c->h_poses[buf], sizeof(double) * 16 * c->batch);
  if (n_edges_out) {
    std::memcpy(n_edges_out, c->h_nedges[buf], sizeof(int) * c->batch);
    if (c->partial[buf])
      for (int l = 0; l < c->batch; ++l) if (!c->stepped[buf][l]) n_edges_out[l] = -1;
  }
  return 0;
}

int liodom_scan_results(liodom_ctx* c, double* poses16_out, int* n_edges_out) {
  return liodom_scan_results_of(c, 0, poses16_out, n_edges_out);
}

int liodom_scan_diag(liodom_ctx* c, int lane, liodom_frame_diag* diag) {
  int rc = check_lane(c, lane); if (rc) return rc;
  if (!diag) return fail(c, LIODOM_E_INVALID, "diag is NULL");
  FrameDiagDev dg;
  CK(cudaMemcpyAsync(&dg, c->d.diag + lane, sizeof(dg), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  diag->n_edges = dg.n_edges;
  for (int k = 0; k < 2; ++k) { diag->n_map[k] = dg.n_map[k]; diag->n_matches[k] = dg.n_matches[k]; copy_summary(dg.solve[k], &diag->solve[k]); }
  std::memcpy(diag->pred_pose, dg.pred_pose, sizeof(dg.pred_pose));
  return 0;
}

int liodom_scan_edges(liodom_ctx* c, int lane, float* edges_xyzi, int cap, int* n_edges) {
  int rc = check_lane(c, lane); if (rc) return rc;
  OdomState os;
  CK(cudaMemcpyAsync(&os, c->d.ostate + lane, sizeof(os), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (n_edges) *n_edges = os.n_edges;
  if (edges_xyzi && os.n_edges > 0) {
    if (cap < os.n_edges) return fail(c, LIODOM_E_CAPACITY, "output capacity %d < %d edges", cap, os.n_edges);
    CK(cudaMemcpy(edges_xyzi, c->d.edges + (size_t)lane * c->d.p.Ecap, (size_t)os.n_edges * 16, cudaMemcpyDeviceToHost));
  }
  return 0;
}

}  // extern "C"
