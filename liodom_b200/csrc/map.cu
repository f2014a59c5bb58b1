// liodom::Map on sm_100a: coarse-cell hash grid with per-cell voxel-centroid clouds (replaces
// src/map.cc:24-189 and include/liodom/map.h:39-116 of the reference).
//
// Reference semantics kept:
//  - updateMap: transform the cloud with the pose (double math, float store), cell key per axis
//    int(floor(p * inv_size) * size + size / 2) (src/map.cc:103-105), find-or-create cells in
//    order of first appearance (:108-118), then re-filter EVERY modified cell with
//    pcl::VoxelGrid(leaf = resolution) over all its points, old centroids counting as single
//    points (:124-128, :56-60).  VoxelGrid output = one centroid per occupied voxel in ascending
//    (z, y, x) lattice order, lattice = floor(p * (1/leaf)) in float (SURVEY.md App. A.3).
//  - getMap: all cells concatenated in creation order (:131-139).
//  - getLocalMap: pose translation truncated to int, (2 cells_xy + 1)^2 cells of the pose's z
//    layer (i outer, j inner) and the z column with the reference's bounds (:141-189).
//
// HBM layout: the whole map is ONE contiguous float4 array in cell-creation order (so getMap is a
// plain copy and a cell is a [offset, count) range); every update rewrites it into the other half
// of a ping-pong pool — touched cells from the sorted work set, untouched cells copied.  At
// 16 B/point that rewrite is HBM-bound and cheap next to the reference's per-cell std::sort.
//
// Touched cells are re-voxelised by a stable LSD radix sort of (touched rank | lattice z | y | x)
// over [old points in stored order..., new points in input order...], so the in-voxel float
// accumulation order is exactly "old centroid first, then new points in arrival order".
#include "../../include/liodom_b200.h"
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

namespace {

constexpr int kTile = 2048;            // keys per radix-sort block (256 threads x 8)
constexpr int kMaxCellVoxels = 1016;   // voxels per axis of one key's points: keeps PCL's per-cell int32 index space (1017^3) from overflowing
constexpr int kRankBits = 16;          // touched-cell rank bits of the sort key (cap_cells = 2^16)
constexpr unsigned long long kEmptyKey = ~0ull;

struct MapState {      // device-resident scalars
  int num_cells;
  int num_points;
  int n_new_slots;
  int n_touched;
  int w_old;           // old points of touched cells
  int n_groups;        // output voxels of touched cells
  int error;           // bit0: coordinate out of packable range, bit1: capacity, bit2: lattice overflow
  int n_dropped;       // non-finite input points (the reference has UB there)
};

struct MapDev {
  double xy, inv_xy, xy_half, zs, inv_z, z_half;
  double xy_slack, z_slack;  // 1 when size / 2 is not an integer (the key's int truncation then moves it up to 1 m), else 0
  float inv_leaf;
  int lat_margin;        // lattice voxels kept below a key's lowest face for float rounding (grows with 1 / resolution)
  int lat_bits;          // bits per lattice axis of the sort key, from the span one key covers; fewer bits = fewer radix passes
  int cap_points, cap_cells, hcap, cap_new;
  float4* pool[2];
  int* cell_count;       // [cap_cells] points per cell (creation order)
  int* cell_off;         // [cap_cells + 1] exclusive prefix of cell_count
  int* cell_newoff;      // [cap_cells + 1]
  int* cell_key;         // [cap_cells][3] reference key ints
  int* touched;          // [cap_cells] 0/1
  int* rank;             // [cap_cells] exclusive prefix of touched
  int* touched_list;     // [cap_cells] cell id per rank
  int* woff;             // [cap_cells + 1] work offsets of old points per rank
  int* group_first;      // [cap_cells + 1] first output group per rank
  unsigned long long* htab;  // [hcap] packed cell key
  int* hval;             // [hcap] cell id
  int* hfirst;           // [hcap] first input index that created the slot (pending cells)
  int* new_slots;        // [cap_new]
  float4* newpts;        // [cap_new] transformed input points
  int* pt_slot;          // [cap_new]
  int* pt_cell;          // [cap_new]
  unsigned long long* keys[2];   // [cap_points + cap_new]
  unsigned* vals[2];
  int* head;             // [cap_points + cap_new] group head flags -> exclusive scan
  int* hist;             // [256 * nblk_max]
  int* scan_tmp;         // block sums of the generic scan
  MapState* st;
  double* pose;          // [12]
};

__device__ __forceinline__ bool pack_key(int kx, int ky, int kz, unsigned long long* out) {
  const int lim = 1 << 20;
  if (kx <= -lim || kx >= lim || ky <= -lim || ky >= lim || kz <= -lim || kz >= lim) return false;
  *out = ((unsigned long long)(unsigned)(kx + lim) << 42) | ((unsigned long long)(unsigned)(ky + lim) << 21) | (unsigned long long)(unsigned)(kz + lim);
  return true;
}
__device__ __forceinline__ unsigned hash_key(unsigned long long k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
  return (unsigned)k;
}
// src/map.cc:103-105, double math then int truncation
__device__ __forceinline__ int cell_key_axis(double v, double inv, double size, double half) {
  return (int)__dadd_rn(__dmul_rn(floor(__dmul_rn(v, inv)), size), half);
}
__device__ __forceinline__ float xform_row(const double* m, double x, double y, double z) {
  return __double2float_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(m[0], x), __dmul_rn(m[1], y)), __dmul_rn(m[2], z)), m[3]));
}
__device__ __forceinline__ int find_slot(const MapDev& m, unsigned long long key) {
  unsigned slot = hash_key(key) & (unsigned)(m.hcap - 1);
  for (;;) {
    const unsigned long long cur = m.htab[slot];
    if (cur == key) return (int)slot;
    if (cur == kEmptyKey) return -1;
    slot = (slot + 1) & (unsigned)(m.hcap - 1);
  }
}

__device__ __forceinline__ int lattice(float v, float inv_leaf) { return (int)floorf(v * inv_leaf); }

// Lattice origin of a key along one axis: the lowest cell face the key can stand for, minus the margin.
// The key int(floor(v / size) * size + size / 2) truncates toward zero, so when size / 2 is not an
// integer a positive key lies up to 1 m below its cell's centre and a non-positive one up to 1 m above
// it; below 2 m the cells -1 and 0 both give key 0, which then covers [-size, size).  The face is taken
// in double: rounding it to float would move it by up to 0.06 m at the edge of the key range.
__device__ __forceinline__ int lattice_origin(int key, double half, double slack, const MapDev& m) {
  const double face = (double)key - half - (key <= 0 ? slack : 0.0);
  return (int)floor(__dmul_rn(face, (double)m.inv_leaf)) - m.lat_margin;
}

// ---------------------------------------------------------------------------------------------------
// Map::updateMap as ONE cooperative launch.  An update touches a few tens of thousands of points, so
// the ~30 dependent launches and two mid-update host round trips of a kernel-per-step pipeline cost more
// than the work; here every step is a grid-stride phase of a single persistent grid (one 256-thread CTA
// per SM) separated by grid-wide barriers, and the sizes that used to travel to the host (touched
// cells, work-set size, number of voxels, radix passes) are read from device memory by every thread.
// ---------------------------------------------------------------------------------------------------
namespace cg = cooperative_groups;
constexpr int kMapThreads = 256;

// exclusive scan of data[0..n) by ONE CTA of 256 threads (8 consecutive items per thread and round)
__device__ void block_scan_excl(int* data, int n, int* total) {
  __shared__ int s_wtot[8];
  __shared__ int s_carry;
  const int tid = threadIdx.x, ln = tid & 31, w = tid >> 5;
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (int base = 0; base < n; base += kMapThreads * 8) {
    int v[8], sum = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { const int i = base + tid * 8 + k; v[k] = i < n ? data[i] : 0; sum += v[k]; }
    int incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (ln >= o) incl += t; }
    if (ln == 31) s_wtot[w] = incl;
    __syncthreads();
    int before = s_carry;
    for (int k = 0; k < w; ++k) before += s_wtot[k];
    int run = before + incl - sum;
#pragma unroll
    for (int k = 0; k < 8; ++k) { const int i = base + tid * 8 + k; if (i < n) data[i] = run; run += v[k]; }
    __syncthreads();
    if (tid == kMapThreads - 1) s_carry = run;
    __syncthreads();
  }
  if (tid == 0 && total) *total = s_carry;
}

// exclusive scan of a long array by the whole grid: chunk sums -> scan of the sums (CTA 0) -> local scans
__device__ void grid_scan_excl(cg::grid_group& grid, int* data, int n, int* tmp, int* total) {
  constexpr int kChunkItems = kMapThreads * 8;
  if (n <= 8 * kChunkItems) {   // short: one CTA does it (the condition is uniform over the grid)
    if (blockIdx.x == 0) block_scan_excl(data, n, total);
    grid.sync();
    return;
  }
  __shared__ int s_w[8];
  const int tid = threadIdx.x, ln = tid & 31, w = tid >> 5;
  const int nchunks = (n + kChunkItems - 1) / kChunkItems;
  for (int c = blockIdx.x; c < nchunks; c += gridDim.x) {
    int sum = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { const int i = c * kChunkItems + tid * 8 + k; if (i < n) sum += data[i]; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (ln == 0) s_w[w] = sum;
    __syncthreads();
    if (tid == 0) { int t = 0; for (int k = 0; k < 8; ++k) t += s_w[k]; tmp[c] = t; }
    __syncthreads();
  }
  grid.sync();
  if (blockIdx.x == 0) block_scan_excl(tmp, nchunks, total);
  grid.sync();
  for (int c = blockIdx.x; c < nchunks; c += gridDim.x) {
    int v[8], sum = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { const int i = c * kChunkItems + tid * 8 + k; v[k] = i < n ? data[i] : 0; sum += v[k]; }
    int incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (ln >= o) incl += t; }
    if (ln == 31) s_w[w] = incl;
    __syncthreads();
    int before = tmp[c];
    for (int k = 0; k < w; ++k) before += s_w[k];
    int run = before + incl - sum;
#pragma unroll
    for (int k = 0; k < 8; ++k) { const int i = c * kChunkItems + tid * 8 + k; if (i < n) data[i] = run; run += v[k]; }
    __syncthreads();
  }
  grid.sync();
}

__global__ void __launch_bounds__(kMapThreads) k_map_update(MapDev m, const float4* in, int n, int cur) {
  cg::grid_group grid = cg::this_grid();
  const int tid = threadIdx.x, ln = tid & 31, w = tid >> 5;
  const int gtid = blockIdx.x * kMapThreads + tid, gsize = gridDim.x * kMapThreads;
  MapState& st = *m.st;
  __shared__ int s_a[kMapThreads], s_b[kMapThreads], s_c[kMapThreads];
  __shared__ int s_carry3[3];
  __shared__ int s_wcnt[8][256];

  // ---- 1: transform, key, find-or-create hash slot (src/map.cc:93-118)
  for (int i = gtid; i < n; i += gsize) {
    const float4 sp = in[i];
    float4 p;
    p.x = xform_row(m.pose, sp.x, sp.y, sp.z); p.y = xform_row(m.pose + 4, sp.x, sp.y, sp.z); p.z = xform_row(m.pose + 8, sp.x, sp.y, sp.z);
    p.w = sp.w;
    m.newpts[i] = p;
    m.pt_slot[i] = -1;
    if (!(isfinite(p.x) && isfinite(p.y) && isfinite(p.z))) { atomicAdd(&st.n_dropped, 1); continue; }
    const int kx = cell_key_axis(p.x, m.inv_xy, m.xy, m.xy_half), ky = cell_key_axis(p.y, m.inv_xy, m.xy, m.xy_half);
    const int kz = cell_key_axis(p.z, m.inv_z, m.zs, m.z_half);
    unsigned long long key;
    if (!pack_key(kx, ky, kz, &key)) { atomicOr(&st.error, 1); continue; }
    unsigned slot = hash_key(key) & (unsigned)(m.hcap - 1);
    for (;;) {
      unsigned long long curk = ((volatile unsigned long long*)m.htab)[slot];
      if (curk == kEmptyKey) {
        curk = atomicCAS(&m.htab[slot], kEmptyKey, key);
        if (curk == kEmptyKey) {  // created: remember it for id assignment
          const int k = atomicAdd(&st.n_new_slots, 1);
          if (k < m.cap_new) m.new_slots[k] = (int)slot; else atomicOr(&st.error, 2);
          curk = key;
        }
      }
      if (curk == key) break;
      slot = (slot + 1) & (unsigned)(m.hcap - 1);
    }
    atomicMin(&m.hfirst[slot], i);
    m.pt_slot[i] = (int)slot;
  }
  grid.sync();

  // ---- 2: new cells get ids in order of first appearance in the input (cells_vector_ order)
  if (gtid == 0) {
    const int nn = min(st.n_new_slots, m.cap_new);
    for (int a = 1; a < nn; ++a) {  // insertion sort by first input index (a handful of cells per update)
      const int sl = m.new_slots[a], f = m.hfirst[sl];
      int b = a - 1;
      while (b >= 0 && m.hfirst[m.new_slots[b]] > f) { m.new_slots[b + 1] = m.new_slots[b]; --b; }
      m.new_slots[b + 1] = sl;
    }
    const int lim = 1 << 20;
    for (int a = 0; a < nn; ++a) {
      const int sl = m.new_slots[a];
      if (st.num_cells >= m.cap_cells) { st.error |= 2; break; }
      const int id = st.num_cells++;
      m.hval[sl] = id;
      const unsigned long long k = m.htab[sl];
      m.cell_key[id * 3 + 0] = (int)((k >> 42) & 0x1fffff) - lim;
      m.cell_key[id * 3 + 1] = (int)((k >> 21) & 0x1fffff) - lim;
      m.cell_key[id * 3 + 2] = (int)(k & 0x1fffff) - lim;
      m.cell_count[id] = 0;
    }
    st.n_new_slots = 0;
  }
  grid.sync();

  // ---- 3: point -> cell id, touched flags
  for (int i = gtid; i < n; i += gsize) {
    const int sl = m.pt_slot[i];
    int cid = -1;
    if (sl >= 0) { cid = m.hval[sl]; if (cid >= 0) m.touched[cid] = 1; }
    m.pt_cell[i] = cid;
  }
  grid.sync();

  // ---- 4 (CTA 0): prefix sums over the cells: old offsets, touched ranks, work offsets
  const int nc = st.num_cells;
  if (blockIdx.x == 0) {
    if (tid < 3) s_carry3[tid] = 0;
    __syncthreads();
    for (int base = 0; base < nc; base += kMapThreads) {
      const int c = base + tid;
      const int cnt = c < nc ? m.cell_count[c] : 0, t = c < nc ? m.touched[c] : 0;
      s_a[tid] = cnt; s_b[tid] = t; s_c[tid] = t ? cnt : 0;
      __syncthreads();
      for (int o = 1; o < kMapThreads; o <<= 1) {
        const int va = tid >= o ? s_a[tid - o] : 0, vb = tid >= o ? s_b[tid - o] : 0, vc = tid >= o ? s_c[tid - o] : 0;
        __syncthreads();
        s_a[tid] += va; s_b[tid] += vb; s_c[tid] += vc;
        __syncthreads();
      }
      if (c < nc) {
        m.cell_off[c] = s_carry3[0] + s_a[tid] - cnt;
        const int r = s_carry3[1] + s_b[tid] - t;
        m.rank[c] = r;
        if (t) { m.touched_list[r] = c; m.woff[r] = s_carry3[2] + s_c[tid] - cnt; }
      }
      __syncthreads();
      if (tid == kMapThreads - 1) { s_carry3[0] += s_a[tid]; s_carry3[1] += s_b[tid]; s_carry3[2] += s_c[tid]; }
      __syncthreads();
    }
    if (tid == 0) {
      m.cell_off[nc] = s_carry3[0];
      m.woff[s_carry3[1]] = s_carry3[2];
      st.n_touched = s_carry3[1];
      st.w_old = s_carry3[2];
    }
  }
  grid.sync();
  const int n_touched = st.n_touched, w_old = st.w_old, wtot = w_old + n, total_old = m.cell_off[nc];

  // ---- 5: sort keys of the work set [old points of touched cells (rank order, stored order) | new points]
  for (int wi = gtid; wi < wtot; wi += gsize) {
    float4 p; int r, cid;
    if (wi < w_old) {
      int lo = 0, hi = n_touched;  // last rank with woff[rank] <= wi
      while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (m.woff[mid] <= wi) lo = mid; else hi = mid; }
      r = lo; cid = m.touched_list[r];
      p = m.pool[cur][m.cell_off[cid] + (wi - m.woff[r])];
    } else {
      const int j = wi - w_old;
      cid = m.pt_cell[j];
      p = m.newpts[j];
      if (cid < 0) { m.keys[0][wi] = kEmptyKey; m.vals[0][wi] = (unsigned)wi; continue; }  // dropped point: sorts last
      r = m.rank[cid];
    }
    // lattice relative to the lowest face the cell's key can stand for
    const int lx = lattice(p.x, m.inv_leaf) - lattice_origin(m.cell_key[cid * 3 + 0], m.xy_half, m.xy_slack, m);
    const int ly = lattice(p.y, m.inv_leaf) - lattice_origin(m.cell_key[cid * 3 + 1], m.xy_half, m.xy_slack, m);
    const int lz = lattice(p.z, m.inv_leaf) - lattice_origin(m.cell_key[cid * 3 + 2], m.z_half, m.z_slack, m);
    const int lim = 1 << m.lat_bits;
    if (lx < 0 || lx >= lim || ly < 0 || ly >= lim || lz < 0 || lz >= lim) atomicOr(&st.error, 4);
    m.keys[0][wi] = ((unsigned long long)r << (3 * m.lat_bits)) | ((unsigned long long)(lz & (lim - 1)) << (2 * m.lat_bits)) |
                    ((unsigned long long)(ly & (lim - 1)) << m.lat_bits) | (unsigned long long)(lx & (lim - 1));
    m.vals[0][wi] = (unsigned)wi;
  }
  grid.sync();

  // ---- stable LSD radix sort, 8-bit digits; key bits in use: 3 * lat_bits lattice bits + ceil(log2(n_touched)).
  // (kEmptyKey = ~0 of dropped points has every processed digit at 255 and no valid key has, so it still sorts last.)
  const int rank_shift = 3 * m.lat_bits;
  int bits = rank_shift;
  while ((1 << (bits - rank_shift)) < n_touched) ++bits;
  const int ntiles = (wtot + kTile - 1) / kTile;
  int sb = 0;
  for (int shift = 0; shift < bits; shift += 8) {
    const unsigned long long* kin = m.keys[sb];
    const unsigned* vin = m.vals[sb];
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      s_a[tid] = 0;
      __syncthreads();
      for (int k = tid; k < kTile; k += kMapThreads) {
        const int i = tile * kTile + k;
        if (i < wtot) atomicAdd(&s_a[(unsigned)(kin[i] >> shift) & 255u], 1);
      }
      __syncthreads();
      m.hist[tid * ntiles + tile] = s_a[tid];
      __syncthreads();
    }
    grid.sync();
    if (blockIdx.x == 0) block_scan_excl(m.hist, 256 * ntiles, nullptr);
    grid.sync();
    unsigned long long* kout = m.keys[sb ^ 1];
    unsigned* vout = m.vals[sb ^ 1];
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {   // each warp owns a contiguous 256-key run, 8 rounds of 32
      for (int k = tid; k < 8 * 256; k += kMapThreads) (&s_wcnt[0][0])[k] = 0;
      __syncthreads();
      int dg[8];
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const int i = tile * kTile + w * 256 + r * 32 + ln;
        const int dgt = i < wtot ? (int)((unsigned)(kin[i] >> shift) & 255u) : -1;
        dg[r] = dgt;
        const unsigned mm = __match_any_sync(0xffffffffu, dgt);
        if (dgt >= 0 && (__ffs(mm) - 1) == ln) s_wcnt[w][dgt] += __popc(mm);
        __syncwarp();
      }
      __syncthreads();
      {
        int run = m.hist[tid * ntiles + tile];
#pragma unroll
        for (int ww = 0; ww < 8; ++ww) { const int c = s_wcnt[ww][tid]; s_wcnt[ww][tid] = run; run += c; }
      }
      __syncthreads();
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const int i = tile * kTile + w * 256 + r * 32 + ln;
        const int dgt = dg[r];
        const unsigned mm = __match_any_sync(0xffffffffu, dgt);
        if (dgt >= 0) {
          const int pos = s_wcnt[w][dgt] + __popc(mm & ((1u << ln) - 1u));
          kout[pos] = kin[i]; vout[pos] = vin[i];
        }
        __syncwarp();
        if (dgt >= 0 && (__ffs(mm) - 1) == ln) s_wcnt[w][dgt] += __popc(mm);
        __syncwarp();
      }
      __syncthreads();
    }
    grid.sync();
    sb ^= 1;
  }
  const unsigned long long* skey = m.keys[sb];
  const unsigned* sval = m.vals[sb];

  // ---- 6: group heads over the sorted keys (a group = one voxel of one touched cell) -> exclusive scan = group index
  for (int wi = gtid; wi < wtot; wi += gsize) {
    const unsigned long long k = skey[wi];
    m.head[wi] = (k != kEmptyKey && (wi == 0 || skey[wi - 1] != k)) ? 1 : 0;
  }
  grid.sync();
  grid_scan_excl(grid, m.head, wtot, m.scan_tmp, &st.n_groups);
  const int n_groups = st.n_groups;

  // first group of every rank; new per-cell counts (touched: its groups; untouched: unchanged)
  for (int r = gtid; r <= n_touched; r += gsize) {
    if (r == n_touched) { m.group_first[r] = n_groups; continue; }
    const unsigned long long target = (unsigned long long)r << rank_shift;
    int lo = 0, hi = wtot;  // first position with key >= target
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (skey[mid] < target) lo = mid + 1; else hi = mid; }
    m.group_first[r] = lo < wtot ? m.head[lo] : n_groups;
  }
  grid.sync();
  for (int c = gtid; c < nc; c += gsize) {
    int cnt = m.cell_count[c];
    if (m.touched[c]) { const int r = m.rank[c]; cnt = m.group_first[r + 1] - m.group_first[r]; }
    m.cell_newoff[c] = cnt;
  }
  grid.sync();
  grid_scan_excl(grid, m.cell_newoff, nc, m.scan_tmp, &m.cell_newoff[nc]);

  // ---- 7: centroids of the touched cells' voxels, sequential float accumulation in sorted order
  // (pcl::CentroidPoint: sum of x, y, z, intensity divided by the count as float); 8: untouched cells move
  for (int wi = gtid; wi < wtot; wi += gsize) {
    const unsigned long long k = skey[wi];
    if (k == kEmptyKey || (wi > 0 && skey[wi - 1] == k)) continue;   // not a group head
    float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
    int cnt = 0;
    for (int u = wi; u < wtot && skey[u] == k; ++u) {
      const int src = (int)sval[u];
      float4 p;
      if (src < w_old) {
        int lo = 0, hi = n_touched;
        while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (m.woff[mid] <= src) lo = mid; else hi = mid; }
        p = m.pool[cur][m.cell_off[m.touched_list[lo]] + (src - m.woff[lo])];
      } else p = m.newpts[src - w_old];
      sx = __fadd_rn(sx, p.x); sy = __fadd_rn(sy, p.y); sz = __fadd_rn(sz, p.z); si = __fadd_rn(si, p.w);
      ++cnt;
    }
    const float fc = (float)cnt;
    const int r = (int)(k >> rank_shift);
    const int g = m.head[wi];   // exclusive scan of the head flags = global group index
    const int cid = m.touched_list[r];
    m.pool[cur ^ 1][m.cell_newoff[cid] + (g - m.group_first[r])] = make_float4(__fdiv_rn(sx, fc), __fdiv_rn(sy, fc), __fdiv_rn(sz, fc), __fdiv_rn(si, fc));
  }
  for (int i = gtid; i < total_old; i += gsize) {
    int lo = 0, hi = nc;  // cell containing old point i
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (m.cell_off[mid] <= i) lo = mid; else hi = mid; }
    if (m.touched[lo]) continue;
    m.pool[cur ^ 1][m.cell_newoff[lo] + (i - m.cell_off[lo])] = m.pool[cur][i];
  }
  grid.sync();

  // ---- commit counts / offsets, reset the per-slot first-index scratch
  for (int c = gtid; c < nc; c += gsize) {
    m.cell_count[c] = m.cell_newoff[c + 1] - m.cell_newoff[c];
    m.cell_off[c] = m.cell_newoff[c];
    m.touched[c] = 0;
  }
  if (gtid == 0) { m.cell_off[nc] = m.cell_newoff[nc]; st.num_points = m.cell_newoff[nc]; }
  for (int i = gtid; i < n; i += gsize)
    if (m.pt_slot[i] >= 0) m.hfirst[m.pt_slot[i]] = INT_MAX;
}

// ---- extraction --------------------------------------------------------------------------------
// Map::getLocalMap in one launch.  keys3: nq < 4096 query keys (reference ints, duplicates allowed).
// Every CTA looks all of them up and scans the counts in shared memory (a few dozen cells: cheaper than
// a grid barrier), then gathers its share of the concatenated cloud.  *total_out = its size; nothing is
// written when it exceeds `cap`.  `out` may be device memory or mapped pinned host memory.
constexpr int kMaxQueryCells = 4096;
__global__ void __launch_bounds__(256) k_map_local(MapDev m, const float4* pool, const int* keys3, int nq, float4* out, int cap, int* total_out) {
  __shared__ int s_off[kMaxQueryCells], s_pre[kMaxQueryCells + 1];
  __shared__ int s_wtot[8];
  const int tid = threadIdx.x, ln = tid & 31, w = tid >> 5;
  constexpr int kPer = kMaxQueryCells / 256;   // consecutive queries per thread
  int cnt[kPer], sum = 0;
#pragma unroll
  for (int k = 0; k < kPer; ++k) {
    const int q = tid * kPer + k;
    int off = 0, c = 0;
    unsigned long long key;
    if (q < nq && pack_key(keys3[q * 3], keys3[q * 3 + 1], keys3[q * 3 + 2], &key)) {
      const int sl = find_slot(m, key);
      if (sl >= 0) { const int cid = m.hval[sl]; if (cid >= 0) { off = m.cell_off[cid]; c = m.cell_count[cid]; } }
    }
    if (q < kMaxQueryCells) s_off[q] = off;
    cnt[k] = c; sum += c;
  }
  int incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (ln >= o) incl += t; }
  if (ln == 31) s_wtot[w] = incl;
  __syncthreads();
  int run = incl - sum;
  for (int k = 0; k < w; ++k) run += s_wtot[k];
#pragma unroll
  for (int k = 0; k < kPer; ++k) { s_pre[tid * kPer + k] = run; run += cnt[k]; }
  if (tid == 255) s_pre[kMaxQueryCells] = run;
  __syncthreads();
  const int total = s_pre[kMaxQueryCells];
  if (blockIdx.x == 0 && tid == 0) *total_out = total;
  if (total > cap || out == nullptr) return;
  for (int i = blockIdx.x * 256 + tid; i < total; i += gridDim.x * 256) {
    int lo = 0, hi = nq;   // last query whose prefix is <= i (empty cells share a prefix: the last one wins, it holds the point)
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (s_pre[mid] <= i) lo = mid; else hi = mid; }
    out[i] = pool[s_off[lo] + (i - s_pre[lo])];
  }
}

}  // namespace

// ===================================================================================================
struct liodom_map {
  MapDev m{};
  int device = 0;
  int cur = 0;
  int nblk_max = 0;
  cudaStream_t stream = nullptr;
  std::vector<void*> allocs;
  std::string err;
  float4* stage_in = nullptr;    // device copy of the input cloud
  int* q_keys = nullptr;         // device scratch of getLocalMap: query keys
  int* q_total = nullptr;        // ... and the size of the gathered cloud
  int* h_total = nullptr;        // pinned
  float* h_gather = nullptr;     // pinned + mapped window the gather kernel writes host results into
  float4* h_gather_dev = nullptr;
  int h_gather_cap = 0;          // points
  std::vector<int> h_keys;
  float4* gather_out = nullptr;  // [cap_points]
  int h_cells = 0, h_points = 0;
  int coop_blocks = 0;           // grid of the cooperative update kernel (every CTA resident)
  long long launches = 0;
};

static thread_local std::string g_map_err;
static int mfail(liodom_map* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof(buf), fmt, ap); va_end(ap);
  if (c) c->err = buf; else g_map_err = buf;
  return code;
}
#define MCK(call)                                                                                  \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) return mfail(c, LIODOM_E_CUDA, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e_)); \
  } while (0)

template <typename T>
static cudaError_t malloc_dev(liodom_map* c, T** p, size_t count, int fill = 0) {
  void* q = nullptr;
  cudaError_t e = cudaMalloc(&q, count * sizeof(T) + 256);
  if (e != cudaSuccess) return e;
  c->allocs.push_back(q);
  e = cudaMemsetAsync(q, fill, count * sizeof(T) + 256, c->stream);
  *p = static_cast<T*>(q);
  return e;
}

extern "C" {

const char* liodom_map_last_error(const liodom_map* m) { return m ? m->err.c_str() : g_map_err.c_str(); }

int liodom_map_create(double voxel_xysize, double voxel_zsize, double resolution, int device, int max_points, liodom_map** out) {
  liodom_map* c = nullptr;
  if (!out || !(voxel_xysize > 0) || !(voxel_zsize > 0) || !(resolution > 0) || max_points < 1)
    return mfail(nullptr, LIODOM_E_INVALID, "bad arguments");
  if (voxel_xysize < 1.0 || voxel_zsize < 1.0)   // the reference's `int += double` cell loops (src/map.cc:157-186) never advance below 1 m
    return mfail(nullptr, LIODOM_E_INVALID, "voxel sizes below 1 m are not supported (the reference's getLocalMap loops do not terminate)");
  // Extent of one key's points per axis: its cell, or the two cells sharing key 0 below 2 m (lattice_origin).
  auto extent = [](double s) { return s < 2.0 ? 2.0 * s : s; };
  auto slack = [](double s) { return s / 2.0 == std::floor(s / 2.0) ? 0.0 : 1.0; };
  const double vox = std::max(extent(voxel_xysize), extent(voxel_zsize)) / resolution;
  if (vox > kMaxCellVoxels)
    return mfail(nullptr, LIODOM_E_INVALID, "cell extent / resolution = %.0f exceeds %d voxels per axis (cells below 2 m count twice: key 0 holds two)",
                 vox, kMaxCellVoxels);
  // A point's float lattice index is off its exact value by at most half an ulp, <= |p| / res * 2^-24 <= 2^20 / res * 2^-24
  // inside the key range; the origin keeps that much + 2 voxels below the lowest face, and the span as much above the top.
  const float inv_leaf = 1.0f / (float)resolution;   // pcl::VoxelGrid: inverse_leaf_size_ in float
  const int margin = 2 + (int)(inv_leaf / 16.0f);
  const double span_m = std::max(extent(voxel_xysize) + slack(voxel_xysize), extent(voxel_zsize) + slack(voxel_zsize));
  const long long span = (long long)std::ceil(span_m * inv_leaf) + 2 * margin + 2;
  int lat_bits = 1;
  while ((1ll << lat_bits) < span) ++lat_bits;
  if (3 * lat_bits + kRankBits > 63)   // kEmptyKey must stay above every sort key
    return mfail(nullptr, LIODOM_E_INVALID, "voxel lattice of %d bits per axis does not fit the 64-bit sort key", lat_bits);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || device < 0 || device >= ndev)
    return mfail(nullptr, LIODOM_E_NODEVICE, "no usable CUDA device (count=%d, requested %d): liodom_b200 has no CPU fallback", ndev, device);
  c = new liodom_map;
  c->device = device;
#define MCC(call)                                                                                  \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      mfail(nullptr, LIODOM_E_CUDA, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e_)); \
      liodom_map_destroy(c);                                                                       \
      return LIODOM_E_CUDA;                                                                        \
    }                                                                                              \
  } while (0)
  MCC(cudaSetDevice(device));
  MCC(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  MapDev& m = c->m;
  m.xy = voxel_xysize; m.inv_xy = 1.0 / voxel_xysize; m.xy_half = voxel_xysize / 2.0;   // src/map.cc:70-81
  m.zs = voxel_zsize; m.inv_z = 1.0 / voxel_zsize; m.z_half = voxel_zsize / 2.0;
  m.xy_slack = slack(voxel_xysize); m.z_slack = slack(voxel_zsize);
  m.inv_leaf = inv_leaf;
  m.lat_margin = margin;
  m.lat_bits = lat_bits;
  m.cap_points = max_points;
  m.cap_new = 1 << 16;
  m.cap_cells = 1 << 16;
  m.hcap = 1 << 18;
  const size_t capw = (size_t)m.cap_points + m.cap_new;
  c->nblk_max = (int)((capw + kTile - 1) / kTile);
  for (int k = 0; k < 2; ++k) {
    MCC(malloc_dev(c, &m.pool[k], (size_t)m.cap_points));
    MCC(malloc_dev(c, &m.keys[k], capw));
    MCC(malloc_dev(c, &m.vals[k], capw));
  }
  MCC(malloc_dev(c, &m.cell_count, (size_t)m.cap_cells));
  MCC(malloc_dev(c, &m.cell_off, (size_t)m.cap_cells + 1));
  MCC(malloc_dev(c, &m.cell_newoff, (size_t)m.cap_cells + 1));
  MCC(malloc_dev(c, &m.cell_key, (size_t)m.cap_cells * 3));
  MCC(malloc_dev(c, &m.touched, (size_t)m.cap_cells));
  MCC(malloc_dev(c, &m.rank, (size_t)m.cap_cells));
  MCC(malloc_dev(c, &m.touched_list, (size_t)m.cap_cells));
  MCC(malloc_dev(c, &m.woff, (size_t)m.cap_cells + 1));
  MCC(malloc_dev(c, &m.group_first, (size_t)m.cap_cells + 1));
  MCC(malloc_dev(c, &m.htab, (size_t)m.hcap, 0xff));
  MCC(malloc_dev(c, &m.hval, (size_t)m.hcap, 0xff));
  MCC(malloc_dev(c, &m.hfirst, (size_t)m.hcap, 0x7f));   // 0x7f7f7f7f > any input index
  MCC(malloc_dev(c, &m.new_slots, (size_t)m.cap_new));
  MCC(malloc_dev(c, &m.newpts, (size_t)m.cap_new));
  MCC(malloc_dev(c, &m.pt_slot, (size_t)m.cap_new));
  MCC(malloc_dev(c, &m.pt_cell, (size_t)m.cap_new));
  MCC(malloc_dev(c, &m.head, capw));
  MCC(malloc_dev(c, &m.hist, (size_t)256 * c->nblk_max));
  MCC(malloc_dev(c, &m.scan_tmp, capw / 2048 + 8));
  MCC(malloc_dev(c, &m.st, 1));
  MCC(malloc_dev(c, &m.pose, 12));
  MCC(malloc_dev(c, &c->stage_in, (size_t)m.cap_new));
  MCC(malloc_dev(c, &c->q_keys, 3 * 4096));
  MCC(malloc_dev(c, &c->q_total, 1));
  MCC(cudaMallocHost(&c->h_total, sizeof(int)));
  c->h_gather_cap = std::min(m.cap_points, 1 << 19);   // 8 MB window; larger local maps take the device path
  MCC(cudaHostAlloc(&c->h_gather, (size_t)c->h_gather_cap * 16, cudaHostAllocMapped));
  { void* dp = nullptr; MCC(cudaHostGetDevicePointer(&dp, c->h_gather, 0)); c->h_gather_dev = static_cast<float4*>(dp); }
  MCC(malloc_dev(c, &c->gather_out, (size_t)m.cap_points));
  {
    int per_sm = 0, sms = 0;
    MCC(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_map_update, kMapThreads, 0));
    MCC(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    if (per_sm < 1) { mfail(nullptr, LIODOM_E_CUDA, "k_map_update cannot be made resident"); liodom_map_destroy(c); return LIODOM_E_CUDA; }
    c->coop_blocks = sms;   // one CTA per SM: the phases are short, more CTAs only lengthen the grid barriers
  }
  MCC(cudaStreamSynchronize(c->stream));
#undef MCC
  *out = c;
  return 0;
}

void liodom_map_destroy(liodom_map* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  for (void* p : c->allocs) cudaFree(p);
  if (c->h_total) cudaFreeHost(c->h_total);
  if (c->h_gather) cudaFreeHost(c->h_gather);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

// Map::updateMap (src/map.cc:90-129): stage the cloud and the pose, ONE cooperative launch, one read-back.
int liodom_map_update(liodom_map* c, const float* pts_xyzi, int n, const double* pose16) {
  if (!c || !pose16 || n < 0) return mfail(c, LIODOM_E_INVALID, "bad arguments");
  MCK(cudaSetDevice(c->device));
  MapDev& m = c->m;
  if (n > m.cap_new) return mfail(c, LIODOM_E_CAPACITY, "cloud of %d points exceeds the per-update capacity %d", n, m.cap_new);
  if (n == 0) return 0;
  if ((size_t)c->h_points + n > (size_t)m.cap_points)
    return mfail(c, LIODOM_E_CAPACITY, "map of %d points + %d new exceeds max_points %d", c->h_points, n, m.cap_points);
  cudaStream_t s = c->stream;
  MCK(cudaMemcpyAsync(c->stage_in, pts_xyzi, (size_t)n * 16, cudaMemcpyHostToDevice, s));
  MCK(cudaMemcpyAsync(m.pose, pose16, sizeof(double) * 12, cudaMemcpyHostToDevice, s));
  const float4* in = c->stage_in;
  int cur = c->cur;
  void* args[] = {(void*)&m, (void*)&in, (void*)&n, (void*)&cur};
  MCK(cudaLaunchCooperativeKernel((const void*)k_map_update, dim3(c->coop_blocks), dim3(kMapThreads), args, 0, s));
  c->launches += 1;
  MapState st;
  MCK(cudaMemcpyAsync(&st, m.st, sizeof(st), cudaMemcpyDeviceToHost, s));
  MCK(cudaStreamSynchronize(s));
  c->cur ^= 1;
  c->h_cells = st.num_cells; c->h_points = st.num_points;
  if (st.error & 1) return mfail(c, LIODOM_E_INVALID, "map coordinates beyond the +-2^20 m key range");
  if (st.error & 2) return mfail(c, LIODOM_E_CAPACITY, "cell capacity exceeded (%d cells)", m.cap_cells);
  if (st.error & 4) return mfail(c, LIODOM_E_INVALID, "voxel lattice overflow inside a cell (cell size / resolution too large)");
  return 0;
}

int liodom_map_size(liodom_map* c, int* n_points, int* n_cells) {
  if (!c) return LIODOM_E_INVALID;
  if (n_points) *n_points = c->h_points;
  if (n_cells) *n_cells = c->h_cells;
  return 0;
}

// Map::getMap (src/map.cc:131-139): the pool already is the concatenation in creation order
int liodom_map_get(liodom_map* c, float* xyzi, int cap, int* n_points) {
  if (!c) return LIODOM_E_INVALID;
  MCK(cudaSetDevice(c->device));
  if (n_points) *n_points = c->h_points;
  if (xyzi && c->h_points > 0) {
    if (cap < c->h_points) return mfail(c, LIODOM_E_CAPACITY, "output capacity %d < map size %d", cap, c->h_points);
    MCK(cudaMemcpyAsync(xyzi, c->m.pool[c->cur], (size_t)c->h_points * 16, cudaMemcpyDeviceToHost, c->stream));
    MCK(cudaStreamSynchronize(c->stream));
  }
  return 0;
}

// Map::getLocalMap (src/map.cc:141-189).  The key list is host integer arithmetic restated from
// the reference (translation truncated to int; the z loop bounds use voxel_xysize_ and `int += double`).
// The cloud is gathered on the device into `dev_out` (capacity `cap` points); returns its size.
static int map_local_keys(liodom_map* c, const double* pose16, int cells_xy, int cells_z, int* nq_out) {
  const MapDev& m = c->m;
  const int x = (int)pose16[3], y = (int)pose16[7], z = (int)pose16[11];
  const int vx = (int)(std::floor(x * m.inv_xy) * m.xy + m.xy_half), vy = (int)(std::floor(y * m.inv_xy) * m.xy + m.xy_half);
  const int vz = (int)(std::floor(z * m.inv_z) * m.zs + m.z_half);
  std::vector<int>& keys = c->h_keys;
  keys.clear();
  const int init_x = (int)(vx - cells_xy * m.xy), end_x = (int)(vx + cells_xy * m.xy);
  const int init_y = (int)(vy - cells_xy * m.xy), end_y = (int)(vy + cells_xy * m.xy);
  for (int i = init_x; i <= end_x && keys.size() < 3 * 4096; i = (int)(i + m.xy))
    for (int j = init_y; j <= end_y && keys.size() < 3 * 4096; j = (int)(j + m.xy)) { keys.push_back(i); keys.push_back(j); keys.push_back(vz); }
  const int init_z = (int)(vz - cells_z * m.xy), end_z = (int)(vz + cells_z * m.xy);
  for (int i = init_z; i <= end_z && keys.size() < 3 * 4096; i = (int)(i + m.zs)) { keys.push_back(vx); keys.push_back(vy); keys.push_back(i); }
  const int nq = (int)keys.size() / 3;
  if (nq >= kMaxQueryCells) return mfail(c, LIODOM_E_CAPACITY, "getLocalMap asks for %d cells (limit %d)", nq, kMaxQueryCells - 1);
  MCK(cudaMemcpyAsync(c->q_keys, keys.data(), sizeof(int) * keys.size(), cudaMemcpyHostToDevice, c->stream));
  *nq_out = nq;
  return 0;
}

// The cloud is gathered into `out` (device memory, or mapped pinned host memory) of capacity `cap` points;
// one launch, one synchronisation.  *n_points = its size even when it does not fit (then nothing is written).
static int map_local_gather(liodom_map* c, const double* pose16, int cells_xy, int cells_z, float4* out, int cap, int* n_points) {
  int nq = 0;
  int rc = map_local_keys(c, pose16, cells_xy, cells_z, &nq);
  if (rc) return rc;
  int blocks = (std::min(c->h_points, std::max(cap, 1)) + 4095) / 4096;
  blocks = std::max(1, std::min(blocks, 148));
  k_map_local<<<blocks, 256, 0, c->stream>>>(c->m, c->m.pool[c->cur], c->q_keys, nq, out, cap, c->q_total);
  c->launches += 1;
  MCK(cudaGetLastError());
  MCK(cudaMemcpyAsync(c->h_total, c->q_total, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  MCK(cudaStreamSynchronize(c->stream));
  if (n_points) *n_points = *c->h_total;
  return 0;
}

int liodom_map_get_local(liodom_map* c, const double* pose16, int cells_xy, int cells_z, float* xyzi, int cap, int* n_points) {
  if (!c || !pose16) return mfail(c, LIODOM_E_INVALID, "bad arguments");
  MCK(cudaSetDevice(c->device));
  int total = 0;
  // first try: straight into the mapped pinned buffer (one launch, one synchronisation, one host memcpy)
  int rc = map_local_gather(c, pose16, cells_xy, cells_z, xyzi ? c->h_gather_dev : nullptr, xyzi ? std::min(cap, c->h_gather_cap) : 0, &total);
  if (rc) return rc;
  if (n_points) *n_points = total;
  if (!xyzi || total == 0) return 0;
  if (cap < total) return mfail(c, LIODOM_E_CAPACITY, "output capacity %d < local map size %d", cap, total);
  if (total <= c->h_gather_cap) { std::memcpy(xyzi, c->h_gather, (size_t)total * 16); return 0; }
  // larger than the pinned window: gather on the device, then copy
  if (total > c->m.cap_points) return mfail(c, LIODOM_E_CAPACITY, "local map of %d points exceeds max_points (duplicated centre cell)", total);
  rc = map_local_gather(c, pose16, cells_xy, cells_z, c->gather_out, c->m.cap_points, &total);
  if (rc) return rc;
  MCK(cudaMemcpyAsync(xyzi, c->gather_out, (size_t)total * 16, cudaMemcpyDeviceToHost, c->stream));
  MCK(cudaStreamSynchronize(c->stream));
  return 0;
}
// Same, but the cloud stays on the device (`dev_xyzi`: device pointer, e.g. the buffer returned by
// liodom_received_map_buffer): the map -> odometry feedback of mapping=1 without a host round trip.
int liodom_map_get_local_device(liodom_map* c, const double* pose16, int cells_xy, int cells_z, void* dev_xyzi, int cap, int* n_points) {
  if (!c || !pose16 || !dev_xyzi) return mfail(c, LIODOM_E_INVALID, "bad arguments");
  MCK(cudaSetDevice(c->device));
  int total = 0;
  const int rc = map_local_gather(c, pose16, cells_xy, cells_z, static_cast<float4*>(dev_xyzi), cap, &total);
  if (rc) return rc;
  if (n_points) *n_points = total;
  if (total > cap) return mfail(c, LIODOM_E_CAPACITY, "output capacity %d < local map size %d", cap, total);
  return 0;
}

int liodom_map_cells(liodom_map* c, int32_t* keys3, int32_t* counts, int cap, int* n_cells) {
  if (!c) return LIODOM_E_INVALID;
  MCK(cudaSetDevice(c->device));
  if (n_cells) *n_cells = c->h_cells;
  if (c->h_cells > 0 && (keys3 || counts)) {
    if (cap < c->h_cells) return mfail(c, LIODOM_E_CAPACITY, "output capacity %d < %d cells", cap, c->h_cells);
    if (keys3) MCK(cudaMemcpyAsync(keys3, c->m.cell_key, sizeof(int) * 3 * c->h_cells, cudaMemcpyDeviceToHost, c->stream));
    if (counts) MCK(cudaMemcpyAsync(counts, c->m.cell_count, sizeof(int) * c->h_cells, cudaMemcpyDeviceToHost, c->stream));
    MCK(cudaStreamSynchronize(c->stream));
  }
  return 0;
}

}  // extern "C"
