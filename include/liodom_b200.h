/* liodom_b200 — C ABI of the B200-native LiODOM hot path.
 *
 * Plain C, plain pointers and sizes; no CUDA, torch, PCL, Eigen or ROS types cross this
 * boundary.  The reference (emiliofidalgo/liodom) has no FFI layer: its boundary is the
 * C++ class surface that src/liodom_node.cc and src/liodom_mapping_node.cc call.  Each
 * entry point below names the reference code it replaces; include/liodom/ holds the
 * C++ facade (same class names) that calls these, and INTEGRATION.md shows the binding.
 *
 * Conventions
 *  - every function returns 0 on success, a negative LIODOM_E_* code otherwise and never
 *    throws; liodom_last_error() gives the message (the reference logs and continues,
 *    SURVEY.md §8(b) "Error conventions").
 *  - points are float32 x,y,z,intensity at the start of each record; `stride_bytes` is
 *    the record size (32 for pcl::PointXYZI, include/liodom/defs.h:35; 16 for packed).
 *  - poses are row-major 4x4 double, world_from_sensor (Eigen::Isometry3d::matrix()).
 *  - a context owns `batch` independent sequences ("lanes"); the reference's single
 *    stream is lane 0 of a batch-1 context.  One context = one worker thread + one CUDA
 *    stream; no re-entrancy (SURVEY.md §8(b) "Threading").
 *  - there is no CPU fallback: if no CUDA device is usable, creation fails.
 */
#ifndef LIODOM_B200_H
#define LIODOM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LIODOM_OK 0
#define LIODOM_E_INVALID -1   /* bad argument / unsupported scan_lines or lidar_type */
#define LIODOM_E_CUDA -2      /* CUDA runtime error (message has the call site) */
#define LIODOM_E_CAPACITY -3  /* input larger than the capacities given at creation */
#define LIODOM_E_NODEVICE -4  /* no usable sm_100 device */

/* Numeric fields of liodom::Params (include/liodom/params.h:33-52; defaults
 * src/params.cc:40-108) plus capacities. */
typedef struct liodom_params {
  double min_range;       /* 3.0 */
  double max_range;       /* 75.0 */
  int lidar_type;         /* 0 Velodyne (ring from elevation), 1 Ouster (ring = row) */
  int scan_lines;         /* 64 (16/32/64 for Velodyne; any <=128 for Ouster) */
  int scan_regions;       /* 8 */
  int edges_per_region;   /* 10 */
  int prev_frames;        /* 5; launch files use 15 (local_map_size_) */
  int filter_local_map;   /* 0 */
  int mapping;            /* 0 */
  int max_points;         /* capacity: points per scan (default 262144) */
  int max_received_map;   /* capacity: points of the received local map (mapping=1) */
  int use_imu;            /* 0; 1: roll/pitch of the predicted pose come from the IMU (src/laser_odometry.cc:152-183) */
} liodom_params;

typedef struct liodom_ctx liodom_ctx;

void liodom_default_params(liodom_params* p);

/* Replaces the FeatureExtractor / LaserOdometer constructors
 * (src/feature_extractor.cc:24-37, src/laser_odometry.cc:71-95). */
int liodom_ctx_create(const liodom_params* p, int batch, int device, liodom_ctx** out);
void liodom_ctx_destroy(liodom_ctx* ctx);
const char* liodom_last_error(const liodom_ctx* ctx); /* ctx may be NULL (creation errors) */
int liodom_max_edges(const liodom_ctx* ctx);          /* scan_lines*scan_regions*(edges_per_region+1) */
void* liodom_stream(const liodom_ctx* ctx);           /* cudaStream_t of the context */
int liodom_sync(liodom_ctx* ctx);

/* ---- FeatureExtractor ------------------------------------------------------------ */

/* splitPointCloud + isValidPoint (src/feature_extractor.cc:84-179), exposed for parity
 * tests.  Host buffers; any output may be NULL.
 *  ring_of_point[n]  ring id or -1;  rings_xyzi[4*n] ring-major stable compaction;
 *  ring_offsets[scan_lines+1];  src_index[n] input index of each compacted point.
 *  n_ambiguous: points whose ring bin is within 1e-12 of a boundary (GPU atan vs libm). */
int liodom_split(liodom_ctx* ctx, int lane, const void* pts, int n, int stride_bytes,
                 int width, int height, int32_t* ring_of_point, float* rings_xyzi,
                 int32_t* ring_offsets, int32_t* src_index, int* n_valid, int* n_ambiguous);

/* Body of FeatureExtractor::operator() (src/feature_extractor.cc:52-59): split +
 * extractFeatures + extractFeaturesFromRegion.  Host in, host out.
 *  edges_xyzi[4*liodom_max_edges()], emitted in (ring, region, pick) order.
 *  Optional debug outputs: edge_ring/edge_idx (ring id and index within the ring),
 *  keys[n_valid] smoothness of every ring-major point (NaN where not evaluated). */
int liodom_extract(liodom_ctx* ctx, int lane, const void* pts, int n, int stride_bytes,
                   int width, int height, float* edges_xyzi, int* n_edges,
                   int32_t* edge_ring, int32_t* edge_idx, double* keys);

/* Where the four FLOAT32 fields of liodom::Point sit inside one point of a sensor_msgs/PointCloud2
 * `data` blob.  Replaces pcl::fromROSMsg in lidarClb / mapClb (src/liodom_node.cc:43-44, :62-63): the
 * message bytes go to the device as they are and the kernels read the fields in place.  The facade's
 * liodom::cloudLayoutFromFields derives it from the message's field list by PCL's rules (match by
 * name, datatype FLOAT32, count 1; a missing intensity stays 0).  point_step need not be a multiple
 * of 4 (the 22-byte velodyne PointXYZIRT works).  Big-endian messages are refused: PCL copies bytes
 * verbatim and would misread them. */
typedef struct liodom_cloud_layout {
  int point_step;     /* PointCloud2.point_step */
  int row_step;       /* PointCloud2.row_step; 0 = width * point_step */
  int off_x, off_y, off_z;
  int off_intensity;  /* < 0: the message has no FLOAT32 "intensity" field */
  int is_bigendian;
} liodom_cloud_layout;

/* liodom_extract on a raw PointCloud2 blob (parity tests of the decode path). */
int liodom_extract_layout(liodom_ctx* ctx, int lane, const void* data, int n, const liodom_cloud_layout* layout,
                          int width, int height, float* edges_xyzi, int* n_edges, int32_t* edge_ring, int32_t* edge_idx);

/* ---- LocalMapManager (src/laser_odometry.cc:24-69) -------------------------------- */
int liodom_lmap_add(liodom_ctx* ctx, int lane, const float* xyzi, int n);
int liodom_lmap_get(liodom_ctx* ctx, int lane, float* xyzi, int cap, int* n_points, int* n_frames);
int liodom_lmap_set_max_frames(liodom_ctx* ctx, int lane, int max_frames);
int liodom_lmap_clear(liodom_ctx* ctx, int lane);
/* SharedData::setLocalMap (src/shared_data.cc:91-96): received local map, mapping=1. */
int liodom_set_received_map(liodom_ctx* ctx, int lane, const float* xyzi, int n);

/* Device-side hand-off of the same cloud: liodom_received_map_buffer gives the lane's device buffer
 * (capacity in points), a producer fills it (liodom_map_get_local_device), liodom_commit_received_map
 * sets its size and rebuilds the voxel hash.  Replaces the ROS hop map_local -> mapClb ->
 * SharedData::setLocalMap (src/liodom_node.cc:57-64) when both processes' work lives on one GPU.
 * liodom_received_map_buffer waits for the context's scans in flight (they read the buffer); the producer must have
 * finished writing (liodom_map_get_local_device synchronises) before liodom_commit_received_map is called, and no
 * liodom_scan_batch may be enqueued between the two calls. */
int liodom_received_map_buffer(liodom_ctx* ctx, int lane, void** dev_xyzi, int* cap);
int liodom_commit_received_map(liodom_ctx* ctx, int lane, int n);

/* ---- LaserOdometer ---------------------------------------------------------------- */
int liodom_odom_reset(liodom_ctx* ctx, int lane);
int liodom_odom_set_pose(liodom_ctx* ctx, int lane, const double* odom16, const double* prev_odom16);
int liodom_odom_get_pose(liodom_ctx* ctx, int lane, double* odom16, double* prev_odom16);

/* use_imu inputs: the latest IMU orientation (x,y,z,w), i.e. SharedData::setLastIMUOri fed by imuClb
 * (src/liodom_node.cc:66-70), and laser_to_base_ as cached by getBaseToLaserTf (src/laser_odometry.cc:368-393;
 * row-major 4x4, identity until set). */
int liodom_odom_set_imu(liodom_ctx* ctx, int lane, const double* q_xyzw);
int liodom_odom_set_laser_to_base(liodom_ctx* ctx, int lane, const double* T16);

typedef struct liodom_solve_summary {
  int iterations;
  int successful_steps;
  int termination;  /* 0 max-iter, 1 gradient tol, 2 parameter tol, 3 function tol, 4 no residuals, 5 failure */
  int num_residual_blocks;
  int cost_evals, jac_evals;
  double initial_cost, final_cost;
} liodom_solve_summary;

typedef struct liodom_frame_diag {
  int n_edges;
  int n_map[2];
  int n_matches[2];
  liodom_solve_summary solve[2];
  double pred_pose[16];
} liodom_frame_diag;

/* addEdgeConstraints up to the residual-block list (src/laser_odometry.cc:300-361)
 * against the lane's current window (+ received map when mapping=1), for parity tests.
 * Per edge: knn_idx[5]/knn_d2[5] (valid when gate bit0 set), gate (bit0: d2[4] < 1.0,
 * bit1: lambda2 > 3*lambda1), eig[3] ascending, q_world[4] transformed edge. */
int liodom_associate(liodom_ctx* ctx, int lane, const float* edges_xyzi, int n_edges,
                     const double* pose16, int32_t* knn_idx, float* knn_d2, uint8_t* gate,
                     double* eig, float* q_world, int* n_map);

/* One ceres::Solve of src/laser_odometry.cc:201-218 on given residual blocks
 * (cab: n x 9 doubles c,a,b).  q = (x,y,z,w), t in/out. */
int liodom_solve(liodom_ctx* ctx, int lane, const double* cab, int n, double* q4, double* t3,
                 liodom_solve_summary* summary);

/* One popFeatures() iteration of LaserOdometer::operator() (src/laser_odometry.cc:108-235):
 * first frame seeds the window; afterwards predict, 2 x {associate, solve}, window update. */
int liodom_register(liodom_ctx* ctx, int lane, const float* edges_xyzi, int n_edges,
                    double* pose16_out, liodom_frame_diag* diag);

/* ---- whole hot path, batched -------------------------------------------------------- */

/* extract + register for every lane in one enqueue.  pts[l] / n[l]: scan of lane l
 * (all with the same stride/width/height).  `on_device` != 0: pts[l] are device pointers
 * (inputs resident in HBM); else host pointers staged through pinned memory.
 * Asynchronous: returns after enqueueing; results are fetched with liodom_scan_results
 * (which synchronises).  Steps may be pipelined: up to 2 scans in flight. */
int liodom_scan_batch(liodom_ctx* ctx, const void* const* pts, const int* n, int stride_bytes,
                      int width, int height, int on_device);
/* Same with raw PointCloud2 blobs: data[l] holds height x row_step bytes (n[l] = width * height points). */
int liodom_scan_batch_layout(liodom_ctx* ctx, const void* const* data, const int* n, const liodom_cloud_layout* layout,
                             int width, int height, int on_device);
/* Step only the listed lanes: lanes[i] takes the scan pts[i] / n[i].  Every other lane's state (pose, window, voxel
 * hash, received map, IMU inputs) is left bit for bit as it was.  Same staging, asynchrony and two-in-flight rules as
 * liodom_scan_batch; host scans back to back in list order go over in one copy.  lanes: any order, no duplicates,
 * each in [0, batch); n_lanes in [0, batch]; n_lanes == 0 enqueues nothing and returns 0.  A bad list returns
 * LIODOM_E_INVALID and enqueues nothing, as does a point-sharded context (it keeps liodom_scan_batch).  The launches
 * are those of a batch-n_lanes context. */
int liodom_scan_lanes(liodom_ctx* ctx, const int32_t* lanes, int n_lanes, const void* const* pts, const int* n,
                      int stride_bytes, int width, int height, int on_device);
int liodom_scan_lanes_layout(liodom_ctx* ctx, const int32_t* lanes, int n_lanes, const void* const* data, const int* n,
                             const liodom_cloud_layout* layout, int width, int height, int on_device);
/* poses16_out[batch*16], n_edges_out[batch] (either may be NULL) of the last enqueued scan.  A lane that step left
 * out (liodom_scan_lanes) reports n_edges = -1 and its last reported pose (zeros if it was never stepped). */
int liodom_scan_results(liodom_ctx* ctx, double* poses16_out, int* n_edges_out);
/* Same for age 0 (last enqueued) or 1 (the scan before it): with two scans in flight the caller
 * enqueues scan k+1, then collects scan k, so the H2D copy of k+1 overlaps the kernels of k.
 * Host input buffers must stay valid until the results of their scan have been collected. */
int liodom_scan_results_of(liodom_ctx* ctx, int age, double* poses16_out, int* n_edges_out);
/* Diagnostics of the last scan of a lane (map sizes, matches, solver summaries); synchronises. */
int liodom_scan_diag(liodom_ctx* ctx, int lane, liodom_frame_diag* diag);
/* Edges of the last scan of a lane (device -> host). */
int liodom_scan_edges(liodom_ctx* ctx, int lane, float* edges_xyzi, int cap, int* n_edges);
/* Number of kernel launches enqueued by this context so far (bench gpu_launches). */
long long liodom_launch_count(const liodom_ctx* ctx);

/* Per-stage device timing of liodom_scan_batch (CUDA events on the context's stream); the
 * counterpart of the reference's Stats timers (src/stats.cc:41-71), with the ring split
 * reported separately (the reference's extraction span excludes it, src/feature_extractor.cc:53-55).
 * Stages: 0 split, 1 extract, 2 predict+associate(outer 0), 3 solve(0), 4 associate(1),
 * 5 solve(1), 6 window update + voxel-hash rebuild. */
#define LIODOM_NUM_STAGES 7
int liodom_stage_timing(liodom_ctx* ctx, int enable);  /* (re)starts accumulation; synchronises */
int liodom_stage_times(liodom_ctx* ctx, double* ms_out /*[LIODOM_NUM_STAGES]*/, int* n_calls);

/* ---- point-sharded mode (BASELINE.json config 5: one large scan across the GPUs of a node) -----
 * Not in the reference (it is single-process CPU).  Extraction shards by ring
 * (src/feature_extractor.cc:186-252 processes rings independently), registration by edge; the
 * window and the LM controller are replicated, so every rank returns the same pose.  Collectives
 * (NCCL, on the context's stream): one all-gather of the edge slots per scan and one all-reduce of
 * 29 doubles per LM evaluation.  One process per GPU; rank 0 creates the id and distributes it
 * (e.g. torch.distributed broadcast); every rank then calls liodom_shard_init on its batch-1
 * context and feeds the SAME scan to liodom_scan_batch.  scan_lines must be a multiple of world. */
int liodom_shard_unique_id(char id_out[128]);
int liodom_shard_init(liodom_ctx* ctx, int rank, int world, const char id[128]);

/* ---- Map (src/map.cc:70-189, include/liodom/map.h:94-116) --------------------------- */
typedef struct liodom_map liodom_map;
int liodom_map_create(double voxel_xysize, double voxel_zsize, double resolution, int device,
                      int max_points, liodom_map** out);
void liodom_map_destroy(liodom_map* m);
const char* liodom_map_last_error(const liodom_map* m);
int liodom_map_update(liodom_map* m, const float* pts_xyzi, int n, const double* pose16);
int liodom_map_size(liodom_map* m, int* n_points, int* n_cells);
int liodom_map_get(liodom_map* m, float* xyzi, int cap, int* n_points);
int liodom_map_get_local(liodom_map* m, const double* pose16, int cells_xy, int cells_z,
                         float* xyzi, int cap, int* n_points);
int liodom_map_cells(liodom_map* m, int32_t* keys3, int32_t* counts, int cap, int* n_cells);
/* getLocalMap with the result left on the device (dev_xyzi: device pointer to cap float4 records). */
int liodom_map_get_local_device(liodom_map* m, const double* pose16, int cells_xy, int cells_z,
                                void* dev_xyzi, int cap, int* n_points);

#ifdef __cplusplus
}
#endif
#endif /* LIODOM_B200_H */
