// Shared device-side layouts and launch prototypes of the liodom_b200 hot path.
//
// HBM layout (per context, B = batch lanes; everything is [lane]-major):
//   scan_in      B x Ncap x stride      staged input scan (host path) or caller memory
//   ring_id      B x Ncap u8            ring of each input point (255 = rejected)
//   chunk_hist   B x chunks x L i32     per-2048-point-chunk ring histogram
//   rings        B x Ncap float4        ring-major stable compaction of the scan
//   ring_off     B x (L+1) i32
//   slots        B x Ecap float4        edges in fixed (ring, region, pick) slots
//   edges        B x Ecap float4        compacted edges (sensor frame)
//   win          B x S x Ecap float4    sliding window slabs (world frame), S = prev_frames+1
//   sorted       B x Mcap float4        window points bucketed by 0.5 m voxel (w = logical index)
//   lin          B x Mcap float4        window (+ received map) in logical order, for neighbour fetches
//   htab         B x Hcap x 16 B        open-addressing voxel hash {key, start, count} (generation tagged)
//   perm         B x Ecap i32           edges in Morton order of their predicted world cell
//   blocks       B x Ecap x 10 f32      residual blocks {c, a, b, valid}
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace liodom {

constexpr int kChunk = 2048;        // points per split chunk (256 threads x 8)
constexpr int kMaxLines = 128;      // scan_lines upper bound
constexpr int kMaxSlots = 64;       // window slabs upper bound (prev_frames + 1)
constexpr int kRingSmemCap = 6144;  // ring points kept in shared memory by k_extract
constexpr unsigned kGenBits = 12;   // hash generation tag width
constexpr unsigned kCntBits = 20;
constexpr int kMaxDynSmem = 227 * 1024;  // opt-in dynamic shared memory per CTA on sm_100
constexpr int kVgTile = 2048;       // keys per CTA of the window-filter radix sort (256 threads x 8)
constexpr int kHashIncr = 0, kHashFullOrdered = 1, kHashFullFast = 2;
constexpr int kPoolFactor = 16;     // bucket pool of the incremental hash, in units of Mcap (a full build uses <= 6, a scan <= 2.2)

// One slot of the open-addressing voxel hash: packed cell key (generation | iz | iy | ix), first
// point of the cell's bucket in `sorted`, and (generation << kCntBits) | points in the cell.
// 16 bytes, so a probe is one 128-bit load.
struct __align__(16) HashEntry {
  unsigned long long key;
  unsigned start;
  unsigned cnt;
};

struct DevParams {
  double min_range, max_range;
  int lidar_type, scan_lines, scan_regions, edges_per_region;
  int prev_frames, filter_local_map, mapping, use_imu;
  int Ncap, Ecap, Mcap, Hcap, Rcap;  // Rcap: received-map capacity
  int Pcap;                          // points of the bucket pool `sorted` (Mcap, or a multiple of it with the incremental hash)
  int LinCap;                        // entries of the ring `lin` (power of two >= Mcap), indexed by sequence number & (LinCap - 1)
  int slots;                         // window slabs allocated
  int chunks;                        // ceil(Ncap / kChunk)
  int batch;
  int Wcap;                          // window capacity in points (slots * Ecap)
  int Bwords;                        // words of the per-lane cell occupancy filter (power of two)
  int vg_blocks;                     // ceil(Wcap / kVgTile) when filter_local_map, else 0
};

// Per-lane description of the scan being processed (rewritten every step).
struct ScanDesc {
  const void* pts;
  int n;
  int stride_bytes;       // point_step
  int width, height;
  // generic sensor_msgs/PointCloud2 layouts (liodom_cloud_layout); generic == 0: x,y,z at 0,4,8 and
  // intensity at +16 (stride >= 32) or +12, rows back to back
  int generic;
  int row_step;           // bytes per row (generic layouts with padded rows), else 0
  int off_x, off_y, off_z, off_i;   // byte offsets of the FLOAT32 fields; off_i < 0: no intensity
};

// Sliding window bookkeeping (LocalMapManager, src/laser_odometry.cc:24-69).
struct WinState {
  int nframes;
  int max_frames;
  int head;               // slab index of the oldest frame
  int total;              // points in the window
  int cnt[kMaxSlots];     // points per slab
  int n_received;         // received local map points (mapping mode)
  unsigned gen;           // hash generation of the current build
  int hash_points;        // points inserted in the current hash build
  int bump;               // bucket allocator
  int n_owners;           // cells created by the current hash build (entries of owner_list)
  // ---- incremental voxel hash (register.cu): the table and the bucket pool persist across scans; a scan evicts
  // the oldest frame's points from the heads of their buckets and appends the new frame's at the tails
  int hmode;              // build chosen by hash_begin: kHashIncr, kHashFullOrdered or kHashFullFast
  int force_full;         // next build must be a full one (host edited the window / tables)
  int built;              // a full ordered build has happened since the last table reset
  int cells_used;         // table slots claimed since the last full build (empty cells stay as tombstones)
  int n_touched;          // cells receiving new points in this build (entries of owner_list)
  unsigned g_next;        // sequence number of the next point entering the window
  unsigned g_base[kMaxSlots];   // sequence number of the first point of the frame in each slab
  int ev_slab, ev_cnt;    // frame evicted by the last commit (ev_cnt 0: none)
  int nw_slab, nw_cnt;    // frame added by the last commit
  unsigned nw_g;          // its first sequence number
  // logical view of the window (oldest frame first), refreshed whenever the window changes:
  int view_prefix[kMaxSlots + 1];   // first logical index of frame k
  int view_slab[kMaxSlots];         // slab holding frame k
  // filter_local_map (computeLocalMap, src/laser_odometry.cc:286-292): VoxelGrid(0.4) of the window
  int vg_active;          // this build's kNN target is the filtered window
  int vg_passes;          // 8-bit radix passes needed for the voxel index range
  int vg_minb[3];         // floor(min * inv_leaf) per axis
  int vg_div[3];          // voxels per axis of the bounding box
  unsigned vg_lo[3];      // ordered-int encoded min / max of the finite window points
  unsigned vg_hi[3];
  unsigned vg_invalid;    // sort key of non-finite points (= number of voxels of the box)
};

// LaserOdometer state (src/laser_odometry.cc: odom_, prev_odom_, param_q, param_t, init_).
struct OdomState {
  double odom[12];        // row-major 3x4
  double prev[12];
  double q[4];            // x,y,z,w
  double t[3];
  int init;
  int frame;
  int n_edges;
  int n_valid;            // valid points of the last split
  int n_ambiguous;
  int pad;
  // use_imu (src/laser_odometry.cc:152-183): latest IMU orientation (x,y,z,w; SharedData::setLastIMUOri)
  // and the cached base->laser transform laser_to_base_ (:368-393), row-major 3x4
  double imu_q[4];
  double l2b[12];
};

struct SolveSummaryDev {
  int iterations, successful_steps, termination, num_residual_blocks, cost_evals, jac_evals;
  double initial_cost, final_cost;
};

struct FrameDiagDev {
  int n_edges;
  int n_map[2];
  int n_matches[2];
  int pad;
  SolveSummaryDev solve[2];
  double pred_pose[16];
};

// Everything the kernels need, passed by value (fits the 4 KB parameter space).
struct DevBuffers {
  DevParams p;
  ScanDesc* scan;          // [B]
  uint8_t* ring_id;        // [B][Ncap]
  int* chunk_hist;         // [B][chunks][L]
  int* chunk_base;         // [B][chunks][L]
  int* chunk_amb;          // [B][chunks] ring-bin decisions within 1e-9 of a boundary
  float4* rings;           // [B][Ncap]
  int* src_index;          // [B][Ncap] (debug) or null
  int* ring_off;           // [B][L+1]
  double* keys;            // [B][Ncap] smoothness (debug output / long-ring path)
  unsigned* pick_bits;     // [B][2][Ncap/32 + kMaxLines + 2] picked bitmaps of the long-ring path
  float4* slots;           // [B][Ecap]
  int* slot_idx;           // [B][Ecap] index within ring of each slot pick
  int* region_cnt;         // [B][L*R]
  float4* edges;           // [B][Ecap]
  int* edge_ring;          // [B][Ecap]
  int* edge_idx;           // [B][Ecap]
  float4* win;             // [B][slots][Ecap]
  float4* received;        // [B][Rcap]
  WinState* wstate;        // [B]
  OdomState* ostate;       // [B]
  float4* sorted;          // [B][Pcap] bucket pool: the points of a voxel are contiguous, oldest frame first; w = sequence number
  float4* lin;             // [B][LinCap] ring of the same points by sequence number (neighbour fetches)
  unsigned* cap_end;       // [B][Hcap] end of the pool region reserved for the cell in each table slot
  unsigned* newcnt;        // [B][Hcap] points of the frame being added per cell (zero between builds)
  unsigned* cell_base;     // [B][Hcap] where this build's new points of the cell go
  HashEntry* htab;         // [B][Hcap]
  unsigned* bloom;         // [B][Bwords] occupancy filter of the hash cells: word = hash(ix >> 5, iy, iz), bit = ix & 31
  unsigned* owner_list;    // [B][Mcap] hash slots of the cells created by the current build
  unsigned* pt_slot;       // [B][Mcap]
  unsigned* pt_rank;       // [B][Mcap]
  int* perm;               // [B][Ecap] Morton-ordered edge indices (thread -> edge) of k_associate
  int* knn_out;            // [B][Ecap][5] neighbours found by k_associate (logical indices, -1: fewer than five within 1 m)
  float* blocks;           // [B][Ecap][10]
  int* knn_idx;            // [B][Ecap][5] (debug) or null
  float* knn_d2;           // [B][Ecap][5]
  uint8_t* gate;           // [B][Ecap]
  double* eig;             // [B][Ecap][3]
  float4* q_world;         // [B][Ecap]
  float4* filtered;        // [B][Wcap] VoxelGrid(0.4) of the window (filter_local_map) or null
  unsigned* vg_key[2];     // [B][Wcap] voxel index of each window point (radix sort ping-pong)
  unsigned* vg_val[2];     // [B][Wcap] logical window index
  int* vg_hist;            // [B][256 * vg_blocks] digit histograms (digit-major)
  int* vg_heads;           // [B][vg_blocks] voxels starting in each tile
  void* shard_ctrl;        // [B] LM controller state of the point-sharded solve (solve.cu)
  double* shard_acc;       // [B][32] partial / reduced normal equations of the point-sharded solve
  FrameDiagDev* diag;      // [B]
  double* poses_out;       // [B][16]
  const int* lanes;        // [n_lanes] lane stepped at each position of a partial step (liodom_scan_lanes); null: identity
};

// Lane at position `pos` of the step's lane list.
__device__ __forceinline__ int lane_at(const DevBuffers& d, int pos) { return d.lanes ? d.lanes[pos] : pos; }

// ---- launchers (each returns the number of kernels it enqueued) ----------------------
// Every kernel works on the lanes at positions [lane0, lane0 + nlanes) of the step's lane list (lane_at); without a
// list (d.lanes null, every single-lane entry point) position and lane coincide.
struct LaneRange { int lane0, nlanes; };
int launch_split(const DevBuffers& d, cudaStream_t s, LaneRange lr);
int launch_extract(const DevBuffers& d, cudaStream_t s, LaneRange lr, bool want_keys);
int launch_hash_build(const DevBuffers& d, cudaStream_t s, LaneRange lr);
int launch_window_filter(const DevBuffers& d, cudaStream_t s, LaneRange lr);   // voxelgrid.cu; 0 launches when the filter is off
int launch_hash_rebuild(const DevBuffers& d, cudaStream_t s, int lane);
int launch_predict(const DevBuffers& d, cudaStream_t s, LaneRange lr);  // + Morton ordering of the edges
int launch_associate(const DevBuffers& d, cudaStream_t s, LaneRange lr, int outer_it, bool force, const double* pose_override);
int launch_solve(const DevBuffers& d, cudaStream_t s, LaneRange lr, int outer_it);
int launch_solve_blocks(const DevBuffers& d, cudaStream_t s, int lane, const double* cab, int n, double* qt_inout,
                        SolveSummaryDev* sum);
int launch_window_update(const DevBuffers& d, cudaStream_t s, LaneRange lr);
int launch_lmap_add(const DevBuffers& d, cudaStream_t s, int lane, const float4* pts_dev, int n);
int launch_lmap_gather(const DevBuffers& d, cudaStream_t s, int lane, float4* out);
int extract_ring_cap(const DevParams& p);
cudaError_t configure_extract_kernels();          // per device, from liodom_ctx_create
size_t extract_smem_needed(const DevParams& p);   // largest dynamic shared memory request of k_extract / k_compact
int launch_extract_rings(const DevBuffers& d, cudaStream_t s, LaneRange lr, int ring0, int nrings);
int launch_compact(const DevBuffers& d, cudaStream_t s, LaneRange lr);
int launch_associate_shard(const DevBuffers& d, cudaStream_t s, int lane, int outer_it, int rank, int world);

// ---- point-sharded mode (shard.cu, solve.cu) -----------------------------------------------------
struct ShardComm { void* comm = nullptr; int rank = 0; int world = 1; };
int shard_unique_id(char out[128]);
int shard_comm_init(ShardComm* sc, int rank, int world, const char id_bytes[128]);
void shard_comm_destroy(ShardComm* sc);
const char* shard_error_string(int rc);
int shard_allreduce_f64(const ShardComm* sc, double* buf, size_t n, cudaStream_t s);
int shard_allgather_bytes(const ShardComm* sc, void* buf, size_t bytes_per_rank, cudaStream_t s);
int shard_group_start();
int shard_group_end();
size_t shard_ctrl_bytes();
int launch_solve_shard(const DevBuffers& d, cudaStream_t s, int lane, int outer_it, const ShardComm* sc, int* nccl_rc);

// ---- small device helpers ---------------------------------------------------------------
__device__ __forceinline__ unsigned long long pack_cell(int ix, int iy, int iz, unsigned gen) {
  return ((unsigned long long)gen << 48) | ((unsigned long long)(iz & 0xFFFF) << 32) |
         ((unsigned long long)(iy & 0xFFFF) << 16) | (unsigned long long)(ix & 0xFFFF);
}
// kNN voxel: 0.5 m (x * 2 is exact in float, so the cell of a point is well defined).  16 bits per
// axis in the packed key: cells alias 32.8 km apart, far beyond the 150 m a window can span.
// (0.25 m cells were measured: 3x fewer candidates per edge, but 18 % instead of 8 % of the edges
// then need the cooperative fallback and the hash build doubles: 0.78 vs 0.46 ms per step.)
constexpr float kCell = 0.5f, kCellInv = 2.0f;
__device__ __forceinline__ int cell_of(float v) { return (int)floorf(v * kCellInv); }
__device__ __forceinline__ unsigned hash_cell(unsigned long long k) {
  // murmur3 fmix64 of the 48-bit cell key: every key bit reaches the low (slot) bits
  k &= 0xFFFFFFFFFFFFull;
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
  return (unsigned)k;
}
// Edge-sharded mode (world > 1 ranks per lane): rank r associates and solves the Morton positions
// [r * share, (r + 1) * share) of the lane's n edges.  A multiple of 32, so every rank starts on a warp boundary.
__host__ __device__ __forceinline__ int edge_share(int n, int world) { return ((n + world - 1) / world + 31) & ~31; }
// word of the occupancy filter holding cell (ix, iy, iz): 32 consecutive cells along x share a word
__device__ __forceinline__ unsigned bloom_word_index(int ixhi, int iy, int iz, unsigned bmask) {
  unsigned h = (unsigned)ixhi * 0x9E3779B1u ^ (unsigned)iy * 0x85EBCA77u ^ (unsigned)iz * 0xC2B2AE3Du;
  h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 12;
  return h & bmask;
}

// ---- logical window addressing -------------------------------------------------------------------
// Frame k (oldest first) lives in slab view_slab[k] and starts at logical index view_prefix[k].  The
// view is kept in WinState (refreshed by hash_begin, i.e. whenever the window changed) so that
// kernels only read it.  `filt` != null: the kNN target is the VoxelGrid-filtered window instead.
struct WinView {
  const int* prefix;
  const int* slab;
  const float4* filt;
  int nframes, total, n_received;
};

__device__ __forceinline__ void load_win_view(const DevBuffers& d, int lane_b, WinView* v, bool target = true) {
  const WinState& ws = d.wstate[lane_b];
  v->prefix = ws.view_prefix; v->slab = ws.view_slab;
  v->nframes = ws.nframes; v->total = ws.view_prefix[ws.nframes];
  v->n_received = d.p.mapping ? ws.n_received : 0;
  v->filt = (target && d.filtered && ws.vg_active) ? d.filtered + (size_t)lane_b * d.p.Wcap : nullptr;
}

__device__ __forceinline__ float4 win_point(const DevBuffers& d, int lane_b, const WinView& v, int i) {
  if (v.filt) return v.filt[i];
  if (i >= v.total) return d.received[(size_t)lane_b * d.p.Rcap + (i - v.total)];
  int lo = 0, hi = v.nframes;   // last frame with prefix <= i
  while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (__ldg(v.prefix + mid) <= i) lo = mid; else hi = mid; }
  return d.win[((size_t)lane_b * d.p.slots + __ldg(v.slab + lo)) * d.p.Ecap + (i - __ldg(v.prefix + lo))];
}

}  // namespace liodom
