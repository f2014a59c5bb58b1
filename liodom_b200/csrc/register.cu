// LaserOdometer data association on sm_100a: sliding window (LocalMapManager), 0.5 m
// open-addressing voxel hash, exact 5-NN, line gate and residual-block assembly
// (replaces src/laser_odometry.cc:24-69, :148-150, :186-195, :231-235, :300-361).
//
// Bit-exact parts (transform, float L2 distances, centroid/scatter/eigen gate) use the
// explicit *_rn intrinsics and the file is compiled with -fmad=false.
#include "common.cuh"
#include <algorithm>
#include <cstdio>
#include <cstdlib>

namespace liodom {

// ---------------------------------------------------------------------------------------
// window addressing
// ---------------------------------------------------------------------------------------
// Called by exactly one thread after the window changed (win_commit) or after the host edited it (force_full):
// refreshes the logical view and chooses how the voxel hash follows the change.
//   kHashIncr         evict the oldest frame's points from the heads of their buckets, append the new frame's at
//                     the tails (table, pool and occupancy filter persist; cost ~ 2 frames instead of the window)
//   kHashFullOrdered  rebuild everything with every bucket in frame order (what kHashIncr needs to start from):
//                     first build, host edits, pool / table / sequence-number headroom used up
//   kHashFullFast     the three-kernel rebuild of the whole target; used when the target is replaced wholesale
//                     every scan anyway (mapping: received map; filter_local_map: VoxelGrid of the window)
__device__ __forceinline__ void hash_begin(const DevBuffers& d, int lane_b, bool force_full = false) {
  WinState& ws = d.wstate[lane_b];
  int acc = 0;
  for (int k = 0; k < ws.nframes; ++k) {
    const int s = (ws.head + k) % d.p.slots;
    ws.view_slab[k] = s; ws.view_prefix[k] = acc; acc += ws.cnt[s];
  }
  ws.view_prefix[ws.nframes] = acc;
  ws.hash_points = ws.total + (d.p.mapping ? ws.n_received : 0);
  // computeLocalMap (src/laser_odometry.cc:286): filter iff the window is full and mapping is off;
  // launch_window_filter then replaces the target (and hash_points) before the hash is built.
  ws.vg_active = (d.filtered && d.p.filter_local_map && !d.p.mapping && ws.nframes == d.p.prev_frames) ? 1 : 0;
  for (int k = 0; k < 3; ++k) { ws.vg_lo[k] = 0xffffffffu; ws.vg_hi[k] = 0u; }
  ws.n_touched = 0;
  const bool fast = d.p.mapping || d.p.filter_local_map;
  // headroom one scan can need in the worst case: every touched cell moves to a region of twice its size
  const long long need = 2ll * ((long long)ws.total + ws.nw_cnt) + 8ll * ws.nw_cnt + 64;
  const bool incr = !fast && !force_full && !ws.force_full && ws.built && (long long)ws.bump + need < (long long)d.p.Pcap &&
                    (long long)ws.cells_used + ws.nw_cnt < (long long)d.p.Hcap / 2 && ws.g_next < 0x70000000u;   // sequence numbers stay non-negative as int (knn_out uses -1 for "none")
  ws.hmode = incr ? kHashIncr : (fast ? kHashFullFast : kHashFullOrdered);
  ws.force_full = 0;
  if (!incr) {
    ws.gen = ws.gen + 1u;     // every entry of the table becomes stale
    ws.bump = 0;
    ws.n_owners = 0;
    ws.cells_used = 0;
    ws.built = fast ? 0 : 1;
    // sequence numbers restart at the logical index (oldest point of the window = 0)
    for (int k = 0; k < ws.nframes; ++k) ws.g_base[ws.view_slab[k]] = (unsigned)ws.view_prefix[k];
    ws.g_next = (unsigned)acc;
  }
}

// LocalMapManager::addPointCloud bookkeeping (src/laser_odometry.cc:34-60): the new frame
// has just been written to slab (head + nframes) % slots with `n` points.
__device__ __forceinline__ void win_commit(const DevBuffers& d, int lane_b, int n) {
  WinState& ws = d.wstate[lane_b];
  const int s = (ws.head + ws.nframes) % d.p.slots;
  ws.cnt[s] = n; ws.total += n; ws.nframes++;
  ws.g_base[s] = ws.g_next; ws.nw_slab = s; ws.nw_cnt = n; ws.nw_g = ws.g_next;
  ws.g_next += (unsigned)n;
  ws.ev_cnt = 0;
  if (ws.nframes > ws.max_frames) {  // drop exactly one (the oldest) frame
    ws.ev_slab = ws.head; ws.ev_cnt = ws.cnt[ws.head];   // its slab stays intact until the ring comes round again
    ws.total -= ws.cnt[ws.head]; ws.cnt[ws.head] = 0;
    ws.head = (ws.head + 1) % d.p.slots; ws.nframes--;
  }
}

// sequence number of the oldest point of the window: logical index = sequence number - this
__device__ __forceinline__ unsigned win_g0(const DevBuffers& d, int lane_b) {
  const WinState& ws = d.wstate[lane_b];
  return ws.nframes > 0 ? ws.g_base[ws.head] : ws.g_next;
}

// ---------------------------------------------------------------------------------------
// voxel hash.  Table: open addressing on packed (ix, iy, iz, generation).  Buckets: contiguous runs of the pool
// `sorted`, the points of a voxel in frame order (oldest first), w = sequence number.  `lin`: ring of the points
// by sequence number.  Three ways to bring it up to date after the window changed (hash_begin picks one):
//   incremental     k_hash_evict_add (eviction + new-frame count, one launch) -> k_hash_grow -> k_hash_add_scatter  (~2 frames of work)
//   full, ordered   k_hash_full_ordered (one CTA per lane; rare)
//   full, fast      k_bloom_clear -> k_hash_insert -> k_hash_alloc -> k_hash_scatter           (mapping / window filter)
// Every kernel returns at once unless its mode is the chosen one, so the host enqueues a fixed sequence.
// ---------------------------------------------------------------------------------------
// Find the table slot of cell `mine` (generation-tagged key), claiming a stale slot if the cell is new.
__device__ __forceinline__ unsigned hash_find_or_create(HashEntry* tab, unsigned mask, unsigned gen, unsigned long long mine, bool* created) {
  unsigned slot = hash_cell(mine) & mask;
  *created = false;
  for (;;) {
    unsigned long long cur = *(volatile unsigned long long*)&tab[slot].key;
    if (cur == mine) break;
    if ((unsigned)(cur >> 48) != gen) {  // stale generation: free
      const unsigned long long prev = atomicCAS(&tab[slot].key, cur, mine);
      if (prev == cur) { *created = true; break; }
      if (prev == mine) break;
      if ((unsigned)(prev >> 48) != gen) continue;  // lost to another stale observer; retry the slot
    }
    slot = (slot + 1) & mask;
  }
  return slot;
}

__device__ __forceinline__ void bloom_publish(const DevBuffers& d, int lane_b, const float4& pt) {
  const int ix = cell_of(pt.x);
  atomicOr(d.bloom + (size_t)lane_b * d.p.Bwords + bloom_word_index(ix >> 5, cell_of(pt.y), cell_of(pt.z), (unsigned)d.p.Bwords - 1u), 1u << (ix & 31));
}

__device__ __forceinline__ void hash_check_generation(const WinState& ws) {
  // The 12-bit tag only distinguishes generations because the host clears the tables and resets ws.gen before it
  // wraps (hash_generation_guard in cabi.cu).  A caller that forgot the guard must fail loudly, not reuse stale cells.
  if (ws.gen >> kGenBits) {
    if (blockIdx.x == 0 && threadIdx.x == 0) printf("liodom_b200: voxel-hash generation %u overflowed its %u-bit tag (missing hash_generation_guard)\n", ws.gen, kGenBits);
    __trap();
  }
}

// ---- full, fast ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_hash_insert(DevBuffers d, int lane0) {
  const int lane_b = lane_at(d, lane0 + blockIdx.y);
  const WinState& ws = d.wstate[lane_b];
  if (ws.hmode != kHashFullFast) return;
  WinView v;
  load_win_view(d, lane_b, &v);
  const int npts = ws.hash_points;
  hash_check_generation(ws);
  const unsigned gen = ws.gen & ((1u << kGenBits) - 1u);
  const unsigned mask = (unsigned)d.p.Hcap - 1u;
  HashEntry* tab = d.htab + (size_t)lane_b * d.p.Hcap;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += gridDim.x * blockDim.x) {
    const float4 pt = win_point(d, lane_b, v, i);
    unsigned* pslot = d.pt_slot + (size_t)lane_b * d.p.Mcap + i;
    if (!(isfinite(pt.x) && isfinite(pt.y) && isfinite(pt.z))) { *pslot = 0xffffffffu; continue; }  // PCL kd-tree skips these
    bool owner;
    const unsigned slot = hash_find_or_create(tab, mask, gen, pack_cell(cell_of(pt.x), cell_of(pt.y), cell_of(pt.z), gen), &owner);
    if (owner) {   // first point of the cell: list it for k_hash_alloc and publish it in the occupancy filter read by k_associate
      d.owner_list[(size_t)lane_b * d.p.Mcap + atomicAdd(&d.wstate[lane_b].n_owners, 1)] = slot;
      bloom_publish(d, lane_b, pt);
    }
    atomicMax(&tab[slot].cnt, gen << kCntBits);
    const unsigned rank = atomicAdd(&tab[slot].cnt, 1u) & ((1u << kCntBits) - 1u);
    *pslot = slot;
    d.pt_rank[(size_t)lane_b * d.p.Mcap + i] = rank;
  }
}

// Bucket allocation: one thread per CELL (the creators appended their slots to owner_list during the insert),
// a warp-wide prefix of the counts and one bump per warp.
__global__ void __launch_bounds__(256) k_hash_alloc(DevBuffers d, int lane0) {
  const int lane_b = lane_at(d, lane0 + blockIdx.y);
  WinState& ws = d.wstate[lane_b];
  if (ws.hmode != kHashFullFast) return;
  const int ncell = ws.n_owners, ln = threadIdx.x & 31;
  HashEntry* tab = d.htab + (size_t)lane_b * d.p.Hcap;
  const unsigned* owners = d.owner_list + (size_t)lane_b * d.p.Mcap;
  const int stride = gridDim.x * blockDim.x;
  for (int j0 = blockIdx.x * blockDim.x + (threadIdx.x & ~31); j0 < ncell; j0 += stride) {   // warp-uniform trip count
    const int j = j0 + ln;
    unsigned slot = 0, cnt = 0;
    if (j < ncell) { slot = owners[j]; cnt = tab[slot].cnt & ((1u << kCntBits) - 1u); }
    unsigned incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned t = __shfl_up_sync(0xffffffffu, incl, o); if (ln >= o) incl += t; }
    unsigned base = 0;
    if (ln == 31) base = (unsigned)atomicAdd(&ws.bump, (int)incl);
    base = __shfl_sync(0xffffffffu, base, 31);
    if (j < ncell) tab[slot].start = base + incl - cnt;
  }
}

__global__ void __launch_bounds__(256) k_hash_scatter(DevBuffers d, int lane0) {
  const int lane_b = lane_at(d, lane0 + blockIdx.y);
  const WinState& ws = d.wstate[lane_b];
  if (ws.hmode != kHashFullFast) return;
  WinView v;
  load_win_view(d, lane_b, &v);
  const int npts = ws.hash_points;
  const HashEntry* tab = d.htab + (size_t)lane_b * d.p.Hcap;
  float4* sorted = d.sorted + (size_t)lane_b * d.p.Pcap;
  float4* lin = d.lin + (size_t)lane_b * d.p.LinCap;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += gridDim.x * blockDim.x) {
    const unsigned ps = d.pt_slot[(size_t)lane_b * d.p.Mcap + i];
    float4 pt = win_point(d, lane_b, v, i);
    lin[i] = pt;                          // sequence number = logical index after a full build
    if (ps == 0xffffffffu) continue;
    pt.w = __int_as_float(i);
    sorted[tab[ps].start + d.pt_rank[(size_t)lane_b * d.p.Mcap + i]] = pt;
  }
}

// Clears the occupancy filters of the lanes (a kernel, not cudaMemsetAsync: a memset may be placed on a
// copy engine, where it would wait behind the next scan's H2D transfer).
__global__ void __launch_bounds__(256) k_bloom_clear(DevBuffers d, int lane0) {
  const int lane_b = lane_at(d, lane0 + blockIdx.y);
  if (d.wstate[lane_b].hmode != kHashFullFast) return;
  uint4* w = reinterpret_cast<uint4*>(d.bloom + (size_t)lane_b * d.p.Bwords);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < d.p.Bwords / 4; i += gridDim.x * blockDim.x) w[i] = make_uint4(0u, 0u, 0u, 0u);
}

// ---- incremental ---------------------------------------------------------------------------------------------
// The evicted frame's points sit at the heads of their buckets (buckets are in frame order): advance the heads.
// Eviction and the new frame's first pass run in ONE launch (even / odd CTAs): both are chains of dependent loads at
// < 25 % issue rate, eviction only touches the (start, count) of cells that exist, the new frame only creates cells and
// counts in `newcnt`, so they commute and their latencies overlap (43 -> ~27 us at 128 lanes).
__device__ __forceinline__ void hash_evict_part(const DevBuffers& d, int lane_b, int part, int nparts) {
  const WinState& ws = d.wstate[lane_b];
  hash_check_generation(ws);
  const unsigned gen = ws.gen & ((1u << kGenBits) - 1u);
  const unsigned mask = (unsigned)d.p.Hcap - 1u;
  HashEntry* tab = d.htab + (size_t)lane_b * d.p.Hcap;
  const float4* slab = d.win + ((size_t)lane_b * d.p.slots + ws.ev_slab) * d.p.Ecap;
  for (int i = part * blockDim.x + threadIdx.x; i < ws.ev_cnt; i += nparts * blockDim.x) {
    const float4 pt = slab[i];
    if (!(isfinite(pt.x) && isfinite(pt.y) && isfinite(pt.z))) continue;   // never inserted
    const unsigned long long key = pack_cell(cell_of(pt.x), cell_of(pt.y), cell_of(pt.z), gen);
    unsigned slot = hash_cell(key) & mask;
    // present by construction (the frame was inserted under this generation); a bounded walk, so that a broken
    // invariant traps instead of hanging the device
    unsigned probes = 0;
    while (*(volatile unsigned long long*)&tab[slot].key != key) {
      slot = (slot + 1) & mask;
      if (++probes > mask) { printf("liodom_b200: evicted point has no voxel-hash cell (lane %d)\n", lane_b); __trap(); }
    }
    atomicAdd(&tab[slot].start, 1u);
    atomicSub(&tab[slot].cnt, 1u);
  }
}

// New frame, pass 1: cell of every point (created if new), rank among the frame's points of that cell.
__device__ __forceinline__ void hash_add_count_part(const DevBuffers& d, int lane_b, int part, int nparts) {
  WinState& ws = d.wstate[lane_b];
  const unsigned gen = ws.gen & ((1u << kGenBits) - 1u);
  const unsigned mask = (unsigned)d.p.Hcap - 1u;
  HashEntry* tab = d.htab + (size_t)lane_b * d.p.Hcap;
  unsigned* newcnt = d.newcnt + (size_t)lane_b * d.p.Hcap;
  const float4* slab = d.win + ((size_t)lane_b * d.p.slots + ws.nw_slab) * d.p.Ecap;
  for (int i = part * blockDim.x + threadIdx.x; i < ws.nw_cnt; i += nparts * blockDim.x) {
    const float4 pt = slab[i];
    unsigned* pslot = d.pt_slot + (size_t)lane_b * d.p.Mcap + i;
    if (!(isfinite(pt.x) && isfinite(pt.y) && isfinite(pt.z))) { *pslot = 0xffffffffu; continue; }
    bool created;
    const unsigned slot = hash_find_or_create(tab, mask, gen, pack_cell(cell_of(pt.x), cell_of(pt.y), cell_of(pt.z), gen), &created);
    if (created) {   // nobody reads start / cnt / cap_end of this slot before k_hash_grow
      tab[slot].start = 0u; tab[slot].cnt = gen << kCntBits;
      d.cap_end[(size_t)lane_b * d.p.Hcap + slot] = 0u;
      bloom_publish(d, lane_b, pt);
      atomicAdd(&ws.cells_used, 1);
    }
    const unsigned rank = atomicAdd(&newcnt[slot], 1u);
    if (rank == 0u) d.owner_list[(size_t)lane_b * d.p.Mcap + atomicAdd(&ws.n_touched, 1)] = slot;
    *pslot = slot;
    d.pt_rank[(size_t)lane_b * d.p.Mcap + i] = rank;
  }
}

__global__ void __launch_bounds__(256) k_hash_evict_add(DevBuffers d, int lane0) {
  const int lane_b = lane_at(d, lane0 + blockIdx.y);
  if (d.wstate[lane_b].hmode != kHashIncr) return;
  const int half = gridDim.x >> 1;   // the grid has an even number of CTAs per lane
  if (blockIdx.x & 1) hash_add_count_part(d, lane_b, blockIdx.x >> 1, half);
  else hash_evict_part(d, lane_b, blockIdx.x >> 1, half);
}

// New frame, pass 2: eight threads per touched cell make room at the tail of its bucket; a bucket that has reached
// the end of its region moves (cooperative copy) to a fresh region of twice its size.  Regions only slide forward —
// heads advance on eviction, tails on insertion — so a steady cell moves once per ~window length of scans.
constexpr int kGrowGroup = 8;
__global__ void __launch_bounds__(256) k_hash_grow(DevBuffers d, int lane0) {
  const int lane_b = lane_at(d, lane0 + blockIdx.y);
  WinState& ws = d.wstate[lane_b];
  if (ws.hmode != kHashIncr) return;
  HashEntry* tab = d.htab + (size_t)lane_b * d.p.Hcap;
  unsigned* newcnt = d.newcnt + (size_t)lane_b * d.p.Hcap;
  unsigned* cap_end = d.cap_end + (size_t)lane_b * d.p.Hcap;
  unsigned* cell_base = d.cell_base + (size_t)lane_b * d.p.Hcap;
  float4* sorted = d.sorted + (size_t)lane_b * d.p.Pcap;
  const unsigned* touched = d.owner_list + (size_t)lane_b * d.p.Mcap;
  const int ln = threadIdx.x & 31, gl = ln & (kGrowGroup - 1), leader = ln & ~(kGrowGroup - 1);
  const unsigned gmask = ((1u << kGrowGroup) - 1u) << leader;
  const int ngroups = gridDim.x * blockDim.x / kGrowGroup, ntouched = ws.n_touched;
  for (int j = (blockIdx.x * blockDim.x + threadIdx.x) / kGrowGroup; j < ntouched; j += ngroups) {   // uniform over a group
    const unsigned slot = touched[j];
    const unsigned nc = newcnt[slot], word = tab[slot].cnt, cnt = word & ((1u << kCntBits) - 1u);
    unsigned start = tab[slot].start;
    if (start + cnt + nc > cap_end[slot]) {
      const unsigned ncap = 2u * (cnt + nc) + 4u;
      unsigned ns = 0;
      if (gl == 0) ns = (unsigned)atomicAdd(&ws.bump, (int)ncap);   // hash_begin guarantees the headroom
      ns = __shfl_sync(gmask, ns, leader);
      for (unsigned k = gl; k < cnt; k += kGrowGroup) sorted[ns + k] = sorted[start + k];
      __syncwarp(gmask);
      if (gl == 0) { tab[slot].start = ns; cap_end[slot] = ns + ncap; }
      start = ns;
    }
    if (gl == 0) { cell_base[slot] = start + cnt; tab[slot].cnt = word + nc; newcnt[slot] = 0u; }
    __syncwarp(gmask);
  }
}

// New frame, pass 3: the points go to the tails of their buckets and into the sequence ring.  The bound keeps 8 CTAs
// per SM (the thread limit): left free, ptxas spends 39 registers on it once the lane comes from the lane list.
__global__ void __launch_bounds__(256, 8) k_hash_add_scatter(DevBuffers d, int lane0) {
  const int lane_b = lane_at(d, lane0 + blockIdx.y);
  const WinState& ws = d.wstate[lane_b];
  if (ws.hmode != kHashIncr) return;
  const unsigned* cell_base = d.cell_base + (size_t)lane_b * d.p.Hcap;
  float4* sorted = d.sorted + (size_t)lane_b * d.p.Pcap;
  float4* lin = d.lin + (size_t)lane_b * d.p.LinCap;
  const unsigned lmask = (unsigned)d.p.LinCap - 1u;
  const float4* slab = d.win + ((size_t)lane_b * d.p.slots + ws.nw_slab) * d.p.Ecap;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < ws.nw_cnt; i += gridDim.x * blockDim.x) {
    float4 pt = slab[i];
    const unsigned g = ws.nw_g + (unsigned)i;
    lin[g & lmask] = pt;
    const unsigned ps = d.pt_slot[(size_t)lane_b * d.p.Mcap + i];
    if (ps == 0xffffffffu) continue;
    pt.w = __uint_as_float(g);
    sorted[cell_base[ps] + d.pt_rank[(size_t)lane_b * d.p.Mcap + i]] = pt;
  }
}

// ---- full, ordered: one CTA per lane, frames scattered oldest first so that every bucket is in frame order ----
constexpr int kFullThreads = 1024;
__global__ void __launch_bounds__(kFullThreads) k_hash_full_ordered(DevBuffers d, int lane0) {
  const int lane_b = lane_at(d, lane0 + blockIdx.x);
  WinState& ws = d.wstate[lane_b];
  if (ws.hmode != kHashFullOrdered) return;
  hash_check_generation(ws);
  const int tid = threadIdx.x;
  const unsigned gen = ws.gen & ((1u << kGenBits) - 1u);
  const unsigned mask = (unsigned)d.p.Hcap - 1u, cmask = (1u << kCntBits) - 1u;
  HashEntry* tab = d.htab + (size_t)lane_b * d.p.Hcap;
  unsigned* cap_end = d.cap_end + (size_t)lane_b * d.p.Hcap;
  unsigned* pt_slot = d.pt_slot + (size_t)lane_b * d.p.Mcap;
  unsigned* owners = d.owner_list + (size_t)lane_b * d.p.Mcap;
  float4* sorted = d.sorted + (size_t)lane_b * d.p.Pcap;
  float4* lin = d.lin + (size_t)lane_b * d.p.LinCap;
  uint4* bw = reinterpret_cast<uint4*>(d.bloom + (size_t)lane_b * d.p.Bwords);
  for (int i = tid; i < d.p.Bwords / 4; i += kFullThreads) bw[i] = make_uint4(0u, 0u, 0u, 0u);
  __syncthreads();
  WinView v;
  load_win_view(d, lane_b, &v, false);
  const int total = v.total;
  // pass 1: cells and their populations
  for (int i = tid; i < total; i += kFullThreads) {
    const float4 pt = win_point(d, lane_b, v, i);
    if (!(isfinite(pt.x) && isfinite(pt.y) && isfinite(pt.z))) { pt_slot[i] = 0xffffffffu; continue; }
    bool created;
    const unsigned slot = hash_find_or_create(tab, mask, gen, pack_cell(cell_of(pt.x), cell_of(pt.y), cell_of(pt.z), gen), &created);
    if (created) { owners[atomicAdd(&ws.n_owners, 1)] = slot; bloom_publish(d, lane_b, pt); }
    atomicMax(&tab[slot].cnt, gen << kCntBits);
    atomicAdd(&tab[slot].cnt, 1u);
    pt_slot[i] = slot;
  }
  __syncthreads();
  // pass 2: a region per cell with room for a few scans of growth; counts restart for the ordered scatter
  const int ncell = ws.n_owners;
  for (int j = tid; j < ncell; j += kFullThreads) {
    const unsigned slot = owners[j], cnt = tab[slot].cnt & cmask, cap = 2u * cnt + 4u;   // first move after ~a window length of scans
    const unsigned start = (unsigned)atomicAdd(&ws.bump, (int)cap);
    tab[slot].start = start; cap_end[slot] = start + cap; tab[slot].cnt = gen << kCntBits;
  }
  if (tid == 0) ws.cells_used = ncell;
  __syncthreads();
  // pass 3: frame after frame (sequence number = logical index, hash_begin renumbered the frames)
  for (int f = 0; f < v.nframes; ++f) {
    const int lo = v.prefix[f], hi = v.prefix[f + 1];
    for (int i = lo + tid; i < hi; i += kFullThreads) {
      float4 pt = win_point(d, lane_b, v, i);
      lin[i] = pt;
      const unsigned slot = pt_slot[i];
      if (slot == 0xffffffffu) continue;
      const unsigned rank = atomicAdd(&tab[slot].cnt, 1u) & cmask;
      pt.w = __int_as_float(i);
      sorted[tab[slot].start + rank] = pt;
    }
    __syncthreads();
  }
}

int launch_hash_build(const DevBuffers& d, cudaStream_t s, LaneRange lr) {
  const int lane0 = lr.lane0, nlanes = lr.nlanes;
  if (d.p.mapping || d.p.filter_local_map) {   // the target is replaced wholesale every scan: full, fast
    int blocks = (d.p.Mcap + 255) / 256;
    if (blocks > 148 * 4) blocks = 148 * 4;
    const dim3 g(blocks, nlanes);
    const int nf = launch_window_filter(d, s, lr);
    k_bloom_clear<<<dim3(std::max(1, std::min(d.p.Bwords / 4 / 256, 64)), nlanes), 256, 0, s>>>(d, lane0);
    k_hash_insert<<<g, 256, 0, s>>>(d, lane0);
    k_hash_alloc<<<g, 256, 0, s>>>(d, lane0);
    k_hash_scatter<<<g, 256, 0, s>>>(d, lane0);
    return 4 + nf;
  }
  const dim3 ge((d.p.Ecap + 255) / 256, nlanes);
  k_hash_full_ordered<<<nlanes, kFullThreads, 0, s>>>(d, lane0);
  k_hash_evict_add<<<dim3(2 * ge.x, ge.y), 256, 0, s>>>(d, lane0);
  k_hash_grow<<<dim3((d.p.Ecap * kGrowGroup / 4 + 255) / 256, nlanes), 256, 0, s>>>(d, lane0);   // ~4 groups' worth of threads per possible cell pair; grid-stride
  k_hash_add_scatter<<<ge, 256, 0, s>>>(d, lane0);
  return 4;
}

// ---------------------------------------------------------------------------------------
// prediction + initial guess (src/laser_odometry.cc:148-150, :186-195). grid B, 32 threads.
// ---------------------------------------------------------------------------------------
__device__ void iso_mul(const double* A, const double* B, double* C) {  // row-major 3x4, implicit last row
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j)
      C[i * 4 + j] = __dadd_rn(__dadd_rn(__dmul_rn(A[i * 4 + 0], B[0 * 4 + j]), __dmul_rn(A[i * 4 + 1], B[1 * 4 + j])), __dmul_rn(A[i * 4 + 2], B[2 * 4 + j]));
    C[i * 4 + 3] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(A[i * 4 + 0], B[3]), __dmul_rn(A[i * 4 + 1], B[7])), __dmul_rn(A[i * 4 + 2], B[11])), A[i * 4 + 3]);
  }
}
__device__ void iso_inverse(const double* A, double* C) {
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) C[i * 4 + j] = A[j * 4 + i];
  for (int i = 0; i < 3; ++i)
    C[i * 4 + 3] = __dadd_rn(__dadd_rn(__dmul_rn(-C[i * 4 + 0], A[3]), __dmul_rn(-C[i * 4 + 1], A[7])), __dmul_rn(-C[i * 4 + 2], A[11]));
}
// Eigen::Quaterniond(Matrix3d) -> (x,y,z,w)
__device__ void quat_from_matrix(const double* A, double* q) {
#define M_(r, c) A[(r) * 4 + (c)]
  const double tr = __dadd_rn(__dadd_rn(M_(0, 0), M_(1, 1)), M_(2, 2));
  if (tr > 0.0) {
    double t = sqrt(__dadd_rn(tr, 1.0));
    q[3] = __dmul_rn(0.5, t); t = __ddiv_rn(0.5, t);
    q[0] = __dmul_rn(__dsub_rn(M_(2, 1), M_(1, 2)), t);
    q[1] = __dmul_rn(__dsub_rn(M_(0, 2), M_(2, 0)), t);
    q[2] = __dmul_rn(__dsub_rn(M_(1, 0), M_(0, 1)), t);
  } else {
    int i = 0;
    if (M_(1, 1) > M_(0, 0)) i = 1;
    if (M_(2, 2) > M_(i, i)) i = 2;
    const int j = (i + 1) % 3, k = (j + 1) % 3;
    double t = sqrt(__dadd_rn(__dsub_rn(__dsub_rn(M_(i, i), M_(j, j)), M_(k, k)), 1.0));
    q[i] = __dmul_rn(0.5, t); t = __ddiv_rn(0.5, t);
    q[3] = __dmul_rn(__dsub_rn(M_(k, j), M_(j, k)), t);
    q[j] = __dmul_rn(__dadd_rn(M_(j, i), M_(i, j)), t);
    q[k] = __dmul_rn(__dadd_rn(M_(k, i), M_(i, k)), t);
  }
#undef M_
}

// ---- use_imu: roll and pitch of the predicted pose (base_link frame) replaced by the IMU's
// (src/laser_odometry.cc:152-183).  tf::Matrix3x3 / tf::Quaternion algebra restated (tf LinearMath,
// third-party): setRotation, getRPY (getEulerYPR solution 1), setRPY (setEulerYPR), getRotation.
__device__ void tf_matrix_from_quat(const double* q /*x,y,z,w*/, double* m /*3x3*/) {
  const double d = q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3];
  const double s = 2.0 / d;
  const double xs = q[0] * s, ys = q[1] * s, zs = q[2] * s;
  const double wx = q[3] * xs, wy = q[3] * ys, wz = q[3] * zs;
  const double xx = q[0] * xs, xy = q[0] * ys, xz = q[0] * zs, yy = q[1] * ys, yz = q[1] * zs, zz = q[2] * zs;
  m[0] = 1.0 - (yy + zz); m[1] = xy - wz; m[2] = xz + wy;
  m[3] = xy + wz; m[4] = 1.0 - (xx + zz); m[5] = yz - wx;
  m[6] = xz - wy; m[7] = yz + wx; m[8] = 1.0 - (xx + yy);
}
__device__ void tf_get_rpy(const double* m, double* roll, double* pitch, double* yaw) {
  const double kPi = 3.14159265358979323846;
  if (fabs(m[6]) >= 1.0) {   // gimbal lock
    *yaw = 0.0;
    if (m[6] < 0.0) { *pitch = kPi / 2.0; *roll = atan2(m[1], m[2]); }
    else { *pitch = -kPi / 2.0; *roll = atan2(-m[1], -m[2]); }
  } else {
    *pitch = -asin(m[6]);
    const double cp = cos(*pitch);
    *roll = atan2(m[7] / cp, m[8] / cp);
    *yaw = atan2(m[3] / cp, m[0] / cp);
  }
}
__device__ void tf_set_rpy(double roll, double pitch, double yaw, double* m) {
  const double ci = cos(roll), cj = cos(pitch), ch = cos(yaw), si = sin(roll), sj = sin(pitch), sh = sin(yaw);
  const double cc = ci * ch, cs = ci * sh, sc = si * ch, ss = si * sh;
  m[0] = cj * ch; m[1] = sj * sc - cs; m[2] = sj * cc + ss;
  m[3] = cj * sh; m[4] = sj * ss + cc; m[5] = sj * cs - sc;
  m[6] = -sj; m[7] = cj * si; m[8] = cj * ci;
}
__device__ void tf_get_rotation(const double* m, double* q /*x,y,z,w*/) {
  const double trace = m[0] + m[4] + m[8];
  if (trace > 0.0) {
    double s = sqrt(trace + 1.0);
    q[3] = s * 0.5; s = 0.5 / s;
    q[0] = (m[7] - m[5]) * s; q[1] = (m[2] - m[6]) * s; q[2] = (m[3] - m[1]) * s;
  } else {
    const int i = m[0] < m[4] ? (m[4] < m[8] ? 2 : 1) : (m[0] < m[8] ? 2 : 0);
    const int j = (i + 1) % 3, k = (i + 2) % 3;
    double s = sqrt(m[i * 3 + i] - m[j * 3 + j] - m[k * 3 + k] + 1.0);
    q[i] = s * 0.5; s = 0.5 / s;
    q[3] = (m[k * 3 + j] - m[j * 3 + k]) * s; q[j] = (m[j * 3 + i] + m[i * 3 + j]) * s; q[k] = (m[k * 3 + i] + m[i * 3 + k]) * s;
  }
}
__device__ void imu_override(OdomState& os) {
  double imu_m[9], r_imu, p_imu, y_imu;
  tf_matrix_from_quat(os.imu_q, imu_m);
  tf_get_rpy(imu_m, &r_imu, &p_imu, &y_imu);
  double bl[12], q[4], m[9], r_bl, p_bl, y_bl;
  iso_mul(os.odom, os.l2b, bl);                  // odom_ * laser_to_base_
  quat_from_matrix(bl, q);                        // Eigen::Quaterniond(odom_bl.rotation())
  tf_matrix_from_quat(q, m);
  tf_get_rpy(m, &r_bl, &p_bl, &y_bl);
  tf_set_rpy(r_imu, p_imu, y_bl, m);
  tf_get_rotation(m, q);
  {  // Eigen::Quaterniond::toRotationMatrix into odom_bl.linear()
    const double x = q[0], y = q[1], z = q[2], w = q[3];
    const double tx = 2.0 * x, ty = 2.0 * y, tz = 2.0 * z;
    const double twx = tx * w, twy = ty * w, twz = tz * w, txx = tx * x, txy = ty * x, txz = tz * x, tyy = ty * y, tyz = tz * y, tzz = tz * z;
    bl[0] = 1.0 - (tyy + tzz); bl[1] = txy - twz; bl[2] = txz + twy;
    bl[4] = txy + twz; bl[5] = 1.0 - (txx + tzz); bl[6] = tyz - twx;
    bl[8] = txz - twy; bl[9] = tyz + twx; bl[10] = 1.0 - (txx + tyy);
  }
  double inv[12], out[12];
  iso_inverse(os.l2b, inv);
  iso_mul(bl, inv, out);                          // odom_bl * laser_to_base_.inverse()
  for (int k = 0; k < 12; ++k) os.odom[k] = out[k];
}

__global__ void k_predict(DevBuffers d, int lane0) {
  const int lane_b = lane_at(d, lane0 + blockIdx.x);
  if (threadIdx.x != 0) return;
  OdomState& os = d.ostate[lane_b];
  FrameDiagDev& dg = d.diag[lane_b];
  dg.n_map[0] = dg.n_map[1] = 0; dg.n_matches[0] = dg.n_matches[1] = 0;
  for (int k = 0; k < 2; ++k) { SolveSummaryDev z = {}; dg.solve[k] = z; }
  if (os.init) {
    double inv[12], rel[12], pred[12];
    iso_inverse(os.prev, inv);
    iso_mul(inv, os.odom, rel);
    iso_mul(os.odom, rel, pred);
    for (int k = 0; k < 12; ++k) { os.prev[k] = os.odom[k]; os.odom[k] = pred[k]; }
    if (d.p.use_imu) imu_override(os);
    quat_from_matrix(os.odom, os.q);
    os.t[0] = os.odom[3]; os.t[1] = os.odom[7]; os.t[2] = os.odom[11];
  }
  for (int k = 0; k < 12; ++k) dg.pred_pose[k] = os.odom[k];
  dg.pred_pose[12] = dg.pred_pose[13] = dg.pred_pose[14] = 0.0; dg.pred_pose[15] = 1.0;
}

// Morton ordering of the edges by the kCell-sized cell of their predicted world position: threads of
// one k_associate warp then walk the same / neighbouring hash buckets (broadcast loads, similar
// trip counts).  Only the thread -> edge assignment changes; outputs stay in edge order.
// One CTA sorts a chunk of kOrderChunk edges in shared memory (bitonic, 64-bit key|index).
constexpr int kOrderChunk = 2048;
__device__ __forceinline__ unsigned spread10(unsigned v) {  // 10 bits -> every third bit
  v &= 0x3ffu;
  v = (v | (v << 16)) & 0x030000ffu;
  v = (v | (v << 8)) & 0x0300f00fu;
  v = (v | (v << 4)) & 0x030c30c3u;
  v = (v | (v << 2)) & 0x09249249u;
  return v;
}
__global__ void __launch_bounds__(1024) k_edge_order(DevBuffers d, int lane0) {
  const DevParams& p = d.p;
  const int lane_b = lane_at(d, lane0 + blockIdx.y);
  const OdomState& os = d.ostate[lane_b];
  const int base = blockIdx.x * kOrderChunk;
  const int n = min(kOrderChunk, os.n_edges - base);
  if (n <= 0) return;
  extern __shared__ unsigned long long sk[];
  int np2 = 64;
  while (np2 < n) np2 <<= 1;
  const float4* edges = d.edges + (size_t)lane_b * p.Ecap + base;
  const float m0 = (float)os.odom[0], m1 = (float)os.odom[1], m2 = (float)os.odom[2], m3 = (float)os.odom[3];
  const float m4 = (float)os.odom[4], m5 = (float)os.odom[5], m6 = (float)os.odom[6], m7 = (float)os.odom[7];
  const float m8 = (float)os.odom[8], m9 = (float)os.odom[9], m10 = (float)os.odom[10], m11 = (float)os.odom[11];
  for (int i = threadIdx.x; i < np2; i += blockDim.x) {
    unsigned long long v = ~0ull;
    if (i < n) {
      const float4 c = edges[i];
      const float x = m0 * c.x + m1 * c.y + m2 * c.z + m3, y = m4 * c.x + m5 * c.y + m6 * c.z + m7, z = m8 * c.x + m9 * c.y + m10 * c.z + m11;
      unsigned key = 0x3fffffffu;  // non-finite edges last
      if (isfinite(x) && isfinite(y) && isfinite(z))
        key = spread10((unsigned)cell_of(x)) | (spread10((unsigned)cell_of(y)) << 1) | (spread10((unsigned)cell_of(z)) << 2);
      v = ((unsigned long long)key << 32) | (unsigned)i;
    }
    sk[i] = v;
  }
  __syncthreads();
  // Bitonic sort (the keys are unique, so the result does not depend on the network).  Every warp owns 64-element
  // blocks; all compare-exchanges at distance j <= 32 stay inside a block, so they run in registers — lane l holds
  // elements l and l + 32 of the block: j = 32 pairs them inside the lane, j <= 16 is a shuffle — and only the
  // distances >= 64 go through shared memory: 15 block-wide stages instead of 66 for 2048 keys.
  const int ln = threadIdx.x & 31, wid = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  auto block_stages = [&](int k, bool from32) {   // the stages j = 32 (if from32) or min(k / 2, 16) ... 1 of merge size k
    for (int b = wid; b < (np2 >> 6); b += nwarps) {
      const int e0 = (b << 6) + ln, e1 = e0 + 32;
      unsigned long long a = sk[e0], c = sk[e1];
      if (from32) {
        const bool asc = (e0 & k) == 0;
        if ((a > c) == asc) { const unsigned long long t = a; a = c; c = t; }
      }
      const bool asc_a = (e0 & k) == 0, asc_c = (e1 & k) == 0;
      for (int j = from32 ? 16 : min(k >> 1, 16); j > 0; j >>= 1) {
        const unsigned long long oa = __shfl_xor_sync(0xffffffffu, a, j), oc = __shfl_xor_sync(0xffffffffu, c, j);
        const bool lower = (ln & j) == 0;
        a = ((lower == asc_a) == (a < oa)) ? a : oa;   // keep the smaller one in the lower position of an ascending pair
        c = ((lower == asc_c) == (c < oc)) ? c : oc;
      }
      sk[e0] = a; sk[e1] = c;
    }
  };
  for (int k = 2; k <= 32; k <<= 1) { block_stages(k, false); }   // (block-local: no barrier needed between them)
  for (int k = 64; k <= np2; k <<= 1) {
    __syncthreads();
    for (int j = k >> 1; j >= 64; j >>= 1) {
      for (int t = threadIdx.x; t < (np2 >> 1); t += blockDim.x) {
        const int lo = ((t & ~(j - 1)) << 1) | (t & (j - 1)), hi = lo | j;
        const unsigned long long a = sk[lo], b = sk[hi];
        const bool up = (lo & k) == 0;
        if ((a > b) == up) { sk[lo] = b; sk[hi] = a; }
      }
      __syncthreads();
    }
    block_stages(k, true);
  }
  __syncthreads();
  int* perm = d.perm + (size_t)lane_b * p.Ecap + base;
  for (int i = threadIdx.x; i < n; i += blockDim.x) perm[i] = base + (int)(unsigned)(sk[i] & 0xffffffffull);
}

int launch_predict(const DevBuffers& d, cudaStream_t s, LaneRange lr) {
  k_predict<<<lr.nlanes, 32, 0, s>>>(d, lr.lane0);
  static_assert(kOrderChunk * 8 <= 48 * 1024, "k_edge_order stays below the 48 KB default: no per-device opt-in needed");
  k_edge_order<<<dim3((d.p.Ecap + kOrderChunk - 1) / kOrderChunk, lr.nlanes), 1024, kOrderChunk * 8, s>>>(d, lr.lane0);
  return 2;
}

// ---------------------------------------------------------------------------------------
// association: one warp per edge. grid (ceil(Ecap/8), nlanes), 256 threads.
// ---------------------------------------------------------------------------------------
// cyclic Jacobi eigenvalues of a symmetric 3x3, +,-,*,/,sqrt only: the same operation
// sequence as the oracle's sym3_eigenvalues (stands in for Eigen::SelfAdjointEigenSolver).
__device__ void sym3_eigenvalues(double a00, double a01, double a02, double a11, double a12, double a22, double* w) {
#define MUL __dmul_rn
#define ADD __dadd_rn
#define SUB __dsub_rn
#define DIV __ddiv_rn
  for (int sweep = 0; sweep < 12; ++sweep) {
    const double off = ADD(ADD(MUL(a01, a01), MUL(a02, a02)), MUL(a12, a12));
    const double diag = ADD(ADD(MUL(a00, a00), MUL(a11, a11)), MUL(a22, a22));
    if (off <= MUL(1e-32, diag) || off == 0.0) break;
    if (a01 != 0.0) {
      const double theta = DIV(SUB(a11, a00), MUL(2.0, a01));
      const double t = DIV(theta >= 0 ? 1.0 : -1.0, ADD(fabs(theta), sqrt(ADD(MUL(theta, theta), 1.0))));
      const double c = DIV(1.0, sqrt(ADD(MUL(t, t), 1.0))), s = MUL(t, c);
      const double n00 = SUB(a00, MUL(t, a01)), n11 = ADD(a11, MUL(t, a01));
      const double n02 = SUB(MUL(c, a02), MUL(s, a12)), n12 = ADD(MUL(s, a02), MUL(c, a12));
      a00 = n00; a11 = n11; a01 = 0.0; a02 = n02; a12 = n12;
    }
    if (a02 != 0.0) {
      const double theta = DIV(SUB(a22, a00), MUL(2.0, a02));
      const double t = DIV(theta >= 0 ? 1.0 : -1.0, ADD(fabs(theta), sqrt(ADD(MUL(theta, theta), 1.0))));
      const double c = DIV(1.0, sqrt(ADD(MUL(t, t), 1.0))), s = MUL(t, c);
      const double n00 = SUB(a00, MUL(t, a02)), n22 = ADD(a22, MUL(t, a02));
      const double n01 = SUB(MUL(c, a01), MUL(s, a12)), n12 = ADD(MUL(s, a01), MUL(c, a12));
      a00 = n00; a22 = n22; a02 = 0.0; a01 = n01; a12 = n12;
    }
    if (a12 != 0.0) {
      const double theta = DIV(SUB(a22, a11), MUL(2.0, a12));
      const double t = DIV(theta >= 0 ? 1.0 : -1.0, ADD(fabs(theta), sqrt(ADD(MUL(theta, theta), 1.0))));
      const double c = DIV(1.0, sqrt(ADD(MUL(t, t), 1.0))), s = MUL(t, c);
      const double n11 = SUB(a11, MUL(t, a12)), n22 = ADD(a22, MUL(t, a12));
      const double n01 = SUB(MUL(c, a01), MUL(s, a02)), n02 = ADD(MUL(s, a01), MUL(c, a02));
      a11 = n11; a22 = n22; a12 = 0.0; a01 = n01; a02 = n02;
    }
  }
  double e0 = a00, e1 = a11, e2 = a22, tmp;
  if (e0 > e1) { tmp = e0; e0 = e1; e1 = tmp; }
  if (e1 > e2) { tmp = e1; e1 = e2; e2 = tmp; }
  if (e0 > e1) { tmp = e0; e0 = e1; e1 = tmp; }
  w[0] = e0; w[1] = e1; w[2] = e2;
}

// Screen of the line gate lambda2 > 3 lambda1 (src/laser_odometry.cc:344) that skips the ~1300 FP64 instructions of the
// Jacobi sweeps for almost every edge: eigenvalues of the symmetric 3x3 from the trigonometric closed form
// (q = tr/3, p = sqrt(|A - qI|_F^2 / 6), r = det((A - qI)/p)/2, phi = acos(r)/3, lambda = q + 2p cos(phi + 2k pi/3)).
// Its error is <= ~1e-8 lambda2 even where two eigenvalues coincide (acos near +-1 amplifies the rounding of r by
// 1/sqrt(eps)); the Jacobi values are within 1e-13 |A| of the true ones.  The decision is taken here only when
// |lambda2 - 3 lambda1| > 1e-5 lambda2, three orders of magnitude beyond both errors, so it is the decision the Jacobi
// values give; otherwise (returns -1: ~1e-5 of the edges, degenerate scatter, NaN) the exact path decides.
// In debug mode (per-edge outputs requested) both run and a disagreement is flagged in the gate byte (bit 2).
__device__ __forceinline__ int sym3_gate_screen(double a00, double a01, double a02, double a11, double a12, double a22) {
  const double q = (a00 + a11 + a22) * (1.0 / 3.0);
  const double b00 = a00 - q, b11 = a11 - q, b22 = a22 - q;
  const double p2 = b00 * b00 + b11 * b11 + b22 * b22 + 2.0 * (a01 * a01 + a02 * a02 + a12 * a12);
  if (!(p2 > 0.0)) return -1;
  const double p = sqrt(p2 * (1.0 / 6.0)), ip = 1.0 / p;
  const double c00 = b00 * ip, c11 = b11 * ip, c22 = b22 * ip, c01 = a01 * ip, c02 = a02 * ip, c12 = a12 * ip;
  double r = 0.5 * (c00 * (c11 * c22 - c12 * c12) - c01 * (c01 * c22 - c12 * c02) + c02 * (c01 * c12 - c11 * c02));
  r = fmin(1.0, fmax(-1.0, r));
  const double phi = acos(r) * (1.0 / 3.0);
  const double l2 = q + 2.0 * p * cos(phi);
  const double l0 = q + 2.0 * p * cos(phi + 2.0943951023931953);
  const double l1 = 3.0 * q - l2 - l0;
  const double dd = l2 - 3.0 * l1, margin = 1e-5 * l2;
  return dd > margin ? 1 : (dd < -margin ? 0 : -1);
}

// A.1: float(m0*x + m1*y + m2*z + m3), double, left to right
__device__ __forceinline__ float xform_row(const double* m, double x, double y, double z) {
  return __double2float_rn(ADD(ADD(ADD(MUL(m[0], x), MUL(m[1], y)), MUL(m[2], z)), m[3]));
}

__device__ __forceinline__ bool cand_less(float d2a, int ia, float d2b, int ib) { return d2a < d2b || (d2a == d2b && ia < ib); }

// Exact 5-NN of one query, one thread per edge, over the kCell = 0.5 m voxel hash.
//
// Exactness.  Every map point with float d2 < (kCell R)^2 lies inside the (2R+1)^3 cell cube
// around the query's cell: an outside point differs by >= kCell R on some axis, and float
// subtraction, squaring and summation are monotone.  So after the 27-cell cube (R = 1) the list is
// final iff its 5th entry has d2 < kCell^2 = 0.25 (92 % of the C1 edges); the others go through
// the fallback stage, which visits every cell of the 5^3 cube (R = 2, radius 1 m) that can still
// hold a candidate — exact for the reference's gate d2[4] < 1.0 (src/laser_odometry.cc:324).
// Pruning.  cell_min_d2 evaluates L2_Simple on the per-axis gaps to the cell box with the same
// float operations as the point distance, hence it is <= the float d2 of every point of the
// cell; a cell is skipped only when that bound is >= 1.0 or strictly above the current 5th
// best, so no candidate (nor a tie on d2, which is broken by the lower logical index) is lost.  A
// whole x-row of cells is skipped on its (y, z) gaps alone: fl(gy^2 + gz^2) <= the bound of each
// of its cells, again by monotonicity.
// Empty cells cost no hash probe: an occupancy filter (one bit per cell, 32 x-consecutive cells per
// word, word = hash(ix >> 5, iy, iz)) is read one row at a time; a false positive costs one probe.
// Sorted 5-list of packed candidates (float bits of d2) << 32 | logical index: d2 >= 0, so the
// unsigned 64-bit order is the (d2, index) order.
struct Knn5 {
  unsigned long long k[5];
};
// Empty entries are (bits of 1.0f) << 32: above every admissible candidate (d2 < 1.0, src/laser_odometry.cc:324 gates on
// the 5th distance), so `key < k[4]` is also the d2 < 1.0 test and an empty list prunes cells beyond the 1 m radius.
constexpr unsigned long long kEmptyCand = 0x3f80000000000000ull;
constexpr float kProvenD2 = kCell * kCell;   // 5th-best below this: the 27-cell cube was enough
constexpr int kFbRadius = (int)(1.0f / kCell);   // cells covering the 1 m gate radius
constexpr int kFbSide = 2 * kFbRadius + 1;

__device__ __forceinline__ float axis_gap(float q, int cell) {
  const float lo = kCell * (float)cell, hi = lo + kCell;   // exact
  // q < lo: lo - q (and q - hi < 0); q > hi: q - hi (and lo - q < 0); inside: both <= 0.  Branch-free; the compiler
  // turned the conditional form into divergent branches inside the neighbour loops.
  return fmaxf(fmaxf(__fsub_rn(lo, q), __fsub_rn(q, hi)), 0.0f);
}

// Sorted insertion of a key known to be below k[4]: four INDEPENDENT comparisons against the old entries, then every
// new entry is a two-level select (8 compare + 16 select instructions; the compare-exchange chain compiled to an LT and
// a GT comparison per stage, 34 instructions, and the insertion is a quarter of the search kernels' instructions).
__device__ __forceinline__ void knn_place(unsigned long long key, unsigned long long* k) {
  const bool c0 = key < k[0], c1 = key < k[1], c2 = key < k[2], c3 = key < k[3];
  const unsigned long long t0 = c0 ? k[0] : key, t1 = c1 ? k[1] : key, t2 = c2 ? k[2] : key, t3 = c3 ? k[3] : key;
  k[4] = t3;
  k[3] = c3 ? t2 : k[3];
  k[2] = c2 ? t1 : k[2];
  k[1] = c1 ? t0 : k[1];
  k[0] = c0 ? key : k[0];
}

__device__ __forceinline__ void knn_offer(const float4& pt, float qx, float qy, float qz, float ub, Knn5& k) {
  // flann::L2_Simple<float>: result += diff*diff over x, y, z in float
  const float ddx = __fsub_rn(qx, pt.x), ddy = __fsub_rn(qy, pt.y), ddz = __fsub_rn(qz, pt.z);
  const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(ddx, ddx), __fmul_rn(ddy, ddy)), __fmul_rn(ddz, ddz));
  const unsigned long long key = ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned)__float_as_int(pt.w);
  if (d2 <= ub && key < k.k[4]) {
    knn_place(key, k.k);
  }
}

// One probe of the voxel hash: {start, count} of the cell's bucket, count 0 if the cell is empty.
__device__ __forceinline__ uint2 hash_lookup(const HashEntry* __restrict__ tab, unsigned hmask, unsigned gen, int ix, int iy, int iz) {
  const unsigned long long key = pack_cell(ix, iy, iz, gen);
  unsigned slot = hash_cell(key) & hmask;
  for (;;) {
    const uint4 e = __ldg(reinterpret_cast<const uint4*>(&tab[slot]));   // key (x,y), start (z), count (w)
    const unsigned long long cur = ((unsigned long long)e.y << 32) | e.x;
    if (cur == key) return make_uint2(e.z, e.w & ((1u << kCntBits) - 1u));
    if ((e.y >> 16) != gen) return make_uint2(0u, 0u);  // free slot: the cell is empty
    slot = (slot + 1) & hmask;
  }
}

// Occupancy bits of the n <= 32 cells ix0 .. ix0 + n - 1 of row (iy, iz); bit b = cell ix0 + b.
__device__ __forceinline__ unsigned bloom_row(const unsigned* __restrict__ bloom, unsigned bmask, int ix0, int n, int iy, int iz) {
  const int w0 = ix0 >> 5, w1 = (ix0 + n - 1) >> 5;
  const unsigned a = __ldg(bloom + bloom_word_index(w0, iy, iz, bmask));
  const unsigned b = w1 != w0 ? __ldg(bloom + bloom_word_index(w1, iy, iz, bmask)) : 0u;
  return __funnelshift_r(a, b, ix0 & 31) & ((1u << n) - 1u);
}

__device__ __forceinline__ float sq_sum2(float gy, float gz) { return __fadd_rn(__fmul_rn(gy, gy), __fmul_rn(gz, gz)); }

__device__ __forceinline__ float cell_min_d2(float qx, float qy, float qz, int ix, int iy, int iz) {
  const float gx = axis_gap(qx, ix), gy = axis_gap(qy, iy), gz = axis_gap(qz, iz);
  return __fadd_rn(__fadd_rn(__fmul_rn(gx, gx), __fmul_rn(gy, gy)), __fmul_rn(gz, gz));
}

__device__ __forceinline__ void knn_scan_bucket(const float4* __restrict__ b, unsigned cn, float qx, float qy, float qz, float ub, Knn5& k) {
  unsigned j = 0;
  for (; j + 4 <= cn; j += 4) {   // four independent loads in flight
    const float4 p0 = __ldg(b + j), p1 = __ldg(b + j + 1), p2 = __ldg(b + j + 2), p3 = __ldg(b + j + 3);
    knn_offer(p0, qx, qy, qz, ub, k); knn_offer(p1, qx, qy, qz, ub, k);
    knn_offer(p2, qx, qy, qz, ub, k); knn_offer(p3, qx, qy, qz, ub, k);
  }
  for (; j < cn; ++j) knn_offer(__ldg(b + j), qx, qy, qz, ub, k);
}

// `ub`: a known upper bound on the final 5th-best d2 (3e38 when none): larger d2 cannot enter.
__device__ __forceinline__ void knn_scan_cell(const HashEntry* __restrict__ tab, const float4* __restrict__ sorted,
                                              unsigned hmask, unsigned gen, int ix, int iy, int iz,
                                              float qx, float qy, float qz, float ub, Knn5& k) {
  const float dmin = cell_min_d2(qx, qy, qz, ix, iy, iz);
  if (__float_as_uint(dmin) > (unsigned)(k.k[4] >> 32) || dmin > ub) return;
  const uint2 sc = hash_lookup(tab, hmask, gen, ix, iy, iz);
  knn_scan_bucket(sorted + sc.x, sc.y, qx, qy, qz, ub, k);
}

// The occupied cells ix0 + b (b < n) of row (iy, iz), except those in `skip`, pruned and scanned.
__device__ __forceinline__ void knn_scan_row(const HashEntry* __restrict__ tab, const float4* __restrict__ sorted,
                                             const unsigned* __restrict__ bloom, unsigned hmask, unsigned bmask, unsigned gen,
                                             int ix0, int n, unsigned skip, int iy, int iz,
                                             float qx, float qy, float qz, float ub, Knn5& k) {
  const float g2 = sq_sum2(axis_gap(qy, iy), axis_gap(qz, iz));
  if (__float_as_uint(g2) > (unsigned)(k.k[4] >> 32) || g2 > ub) return;
  unsigned mask = bloom_row(bloom, bmask, ix0, n, iy, iz) & ~skip;
  while (mask) {
    const int bsel = __ffs(mask) - 1;
    mask &= mask - 1;
    knn_scan_cell(tab, sorted, hmask, gen, ix0 + bsel, iy, iz, qx, qy, qz, ub, k);
  }
}

// Fallback of the 5-NN search: edges whose 5th neighbour is not proven inside the kCell radius.  The whole warp
// walks the 25 x-rows of the owner's 5^3 cube (one row per lane; rows and cells beyond the owner's current 5th
// best or the 1 m gate are skipped on their bounds, the 27 cells of level 1 are masked out), then the per-lane
// lists are merged by 5 rounds of warp arg-min.  Must be called by all 32 lanes; `want`: this lane owns a query.
__device__ __forceinline__ void knn_fallback_warp(const HashEntry* __restrict__ tab, const float4* __restrict__ sorted,
                                                  const unsigned* __restrict__ bloom, unsigned hmask, unsigned bmask, unsigned gen,
                                                  bool want, float qx, float qy, float qz, int cx, int cy, int cz, Knn5& k, int ln) {
  unsigned need = __ballot_sync(0xffffffffu, want && (unsigned)(k.k[4] >> 32) >= __float_as_uint(kProvenD2));
  while (need) {
    const int owner = __ffs(need) - 1;
    need &= need - 1;
    const float jx = __shfl_sync(0xffffffffu, qx, owner), jy = __shfl_sync(0xffffffffu, qy, owner), jz = __shfl_sync(0xffffffffu, qz, owner);
    const int jcx = __shfl_sync(0xffffffffu, cx, owner), jcy = __shfl_sync(0xffffffffu, cy, owner), jcz = __shfl_sync(0xffffffffu, cz, owner);
    const unsigned ubb = __shfl_sync(0xffffffffu, (unsigned)(k.k[4] >> 32), owner);
    const float ub = __uint_as_float(ubb);   // 1.0 when the list is not full yet
    Knn5 l;
#pragma unroll
    for (int r = 0; r < 5; ++r) {   // lane 0 inherits the owner's list, the others start empty
      const unsigned long long v = __shfl_sync(0xffffffffu, k.k[r], owner);
      l.k[r] = ln == 0 ? v : kEmptyCand;
    }
    for (int rr = ln; rr < kFbSide * kFbSide; rr += 32) {
      const int dy = rr % kFbSide - kFbRadius, dz = rr / kFbSide - kFbRadius;
      const unsigned inner = (abs(dy) <= 1 && abs(dz) <= 1) ? (7u << (kFbRadius - 1)) : 0u;
      knn_scan_row(tab, sorted, bloom, hmask, bmask, gen, jcx - kFbRadius, kFbSide, inner, jcy + dy, jcz + dz, jx, jy, jz, ub, l);
    }
    __syncwarp();
#pragma unroll
    for (int r = 0; r < 5; ++r) {   // warp arg-min on the 64-bit heads: high word, then low word among ties
      const unsigned hh = (unsigned)(l.k[0] >> 32), hl = (unsigned)l.k[0];
      const unsigned mh = __reduce_min_sync(0xffffffffu, hh);
      const unsigned ml = __reduce_min_sync(0xffffffffu, hh == mh ? hl : 0xffffffffu);
      const int wl = __ffs(__ballot_sync(0xffffffffu, hh == mh && hl == ml)) - 1;
      if (ln == owner) k.k[r] = ((unsigned long long)mh << 32) | ml;
      if (ln == wl) {
#pragma unroll
        for (int q = 0; q < 4; ++q) l.k[q] = l.k[q + 1];
        l.k[4] = kEmptyCand;
      }
    }
  }
}

// Line gate and residual block of one edge (src/laser_odometry.cc:324-361): centroid and scatter of the five
// neighbours in double, eigenvalues, lambda2 > 3 lambda1, block {c, a, b, valid}.  nn_idx[0] < 0: fewer than five
// neighbours within 1 m.  Returns true when the edge yields a residual block.
__device__ __forceinline__ bool line_gate(const DevBuffers& d, int lane_b, int e, const float4& c, const int* nn_idx) {
  const DevParams& p = d.p;
  uint8_t gt = 0;
  double ev[3] = {0.0, 0.0, 0.0};
  float4 a = make_float4(0, 0, 0, 0), b = make_float4(0, 0, 0, 0);
  if (nn_idx[0] >= 0) {  // five neighbours with d2 < 1.0 (src/laser_odometry.cc:324)
    gt |= 1;
    const float4* lin = d.lin + (size_t)lane_b * p.LinCap;   // ring by sequence number
    const unsigned lmask = (unsigned)p.LinCap - 1u;
    float4 nn[5];
#pragma unroll
    for (int r = 0; r < 5; ++r) nn[r] = lin[(unsigned)nn_idx[r] & lmask];
    // centroid and scatter in double, neighbour order (src/laser_odometry.cc:325-340)
    double mx = 0.0, my = 0.0, mz = 0.0;
#pragma unroll
    for (int r = 0; r < 5; ++r) { mx = ADD(mx, (double)nn[r].x); my = ADD(my, (double)nn[r].y); mz = ADD(mz, (double)nn[r].z); }
    mx = DIV(mx, 5.0); my = DIV(my, 5.0); mz = DIV(mz, 5.0);
    double c00 = 0, c01 = 0, c02 = 0, c11 = 0, c12 = 0, c22 = 0;
#pragma unroll
    for (int r = 0; r < 5; ++r) {
      const double dx = SUB((double)nn[r].x, mx), dy = SUB((double)nn[r].y, my), dz = SUB((double)nn[r].z, mz);
      c00 = ADD(c00, MUL(dx, dx)); c01 = ADD(c01, MUL(dx, dy)); c02 = ADD(c02, MUL(dx, dz));
      c11 = ADD(c11, MUL(dy, dy)); c12 = ADD(c12, MUL(dy, dz)); c22 = ADD(c22, MUL(dz, dz));
    }
    const int screen = sym3_gate_screen(c00, c01, c02, c11, c12, c22);
    bool pass = screen == 1;
    if (screen < 0 || d.gate) {
      sym3_eigenvalues(c00, c01, c02, c11, c12, c22, ev);
      pass = ev[2] > MUL(3.0, ev[1]);   // :344
      if (screen >= 0 && (screen == 1) != pass) gt |= 4;   // debug: the screen must never disagree
    }
    if (pass) { gt |= 2; a = nn[0]; b = nn[1]; }  // :351-357
  }
  float* blk = d.blocks + ((size_t)lane_b * p.Ecap + e) * 10;
  blk[0] = c.x; blk[1] = c.y; blk[2] = c.z; blk[3] = a.x; blk[4] = a.y; blk[5] = a.z;
  blk[6] = b.x; blk[7] = b.y; blk[8] = b.z; blk[9] = (gt & 2) ? 1.0f : 0.0f;
  if (d.gate) {
    const size_t o = (size_t)lane_b * p.Ecap + e;
    d.gate[o] = gt;
    d.eig[o * 3] = ev[0]; d.eig[o * 3 + 1] = ev[1]; d.eig[o * 3 + 2] = ev[2];
  }
  return (gt & 2) != 0;
}

constexpr int kAssocThreads = 64;
constexpr int kAssocMinBlocks1 = 20;   // k_associate<1>: 20 CTAs of kAssocThreads per SM, i.e. at most 48 registers

// Per-edge debug outputs (called when d.gate is set): the five neighbours as logical window indices, their d2, the query.
__device__ __forceinline__ void knn_debug_out(const DevBuffers& d, int lane_b, int e, const Knn5& k, float qx, float qy, float qz, float w) {
  const size_t o = (size_t)lane_b * d.p.Ecap + e;
  for (int r = 0; r < 5; ++r) {
    d.knn_idx[o * 5 + r] = k.k[r] == kEmptyCand ? -1 : (int)((unsigned)k.k[r] - win_g0(d, lane_b));   // logical index
    d.knn_d2[o * 5 + r] = k.k[r] == kEmptyCand ? __int_as_float(0x7f800000) : __uint_as_float((unsigned)(k.k[r] >> 32));
  }
  d.q_world[o] = make_float4(qx, qy, qz, w);
}

// Visit order of the 27 cells of a cube, nearest first: per axis the own cell, then the neighbour behind the nearer face,
// then the one behind the farther face; slots sorted by the sum of the per-axis weights (0, 1, 4): own; one near (3);
// two near (3); three near; one far (3); one far + one near (6); one far + two near (3); two far (3); two far + one
// near (3); three far.  The bound tightens before the far cells are looked at and most of them fall to cell_min_d2.
// The order is applied to the CANONICAL occupancy word: occ_canonical reflects every axis whose near side is +1, so that
// "near" is offset -1 for every lane and slot i is one constant bit, bit = ((cz+1)*3 + (cy+1))*3 + (cx+1) with c = 0
// (own), -1 (near), +1 (far).  The slot test is then two instructions and the offsets are decoded only for occupied
// slots, by arithmetic (a per-slot ?: decode compiled to indirect branches and was 10 % of k_associate<1>).
__constant__ unsigned kNearMask[27] = {
    0x0002000, 0x0001000, 0x0000400, 0x0000010, 0x0000200, 0x0000008, 0x0000002, 0x0000001, 0x0004000,
    0x0010000, 0x0400000, 0x0000800, 0x0008000, 0x0000020, 0x0000080, 0x0200000, 0x0080000, 0x0000004,
    0x0000040, 0x0040000, 0x0020000, 0x0800000, 0x2000000, 0x0000100, 0x0100000, 0x1000000, 0x4000000};
// Cell offsets of slot i: canonical (0 own, -1 near, +1 far; 2-bit two's complement fields x | y << 2 | z << 4) times the
// lane's near direction.  Arithmetic only (the ?: form of the decode compiled to indirect branches).
__constant__ unsigned char kNearOff[27] = {0, 3, 12, 48, 15, 51, 60, 63, 1, 4, 16, 13, 7, 49, 52, 19, 28, 61, 55, 31, 5, 17, 20, 53, 29, 23, 21};
__device__ __forceinline__ void near_offsets(int i, int nx, int ny, int nz, int* dx, int* dy, int* dz) {
  const int v = kNearOff[i];
  *dx = -(((v << 30) >> 30) * nx);
  *dy = -(((v << 28) >> 30) * ny);
  *dz = -(((v << 26) >> 30) * nz);
}
__device__ __forceinline__ unsigned occ_canonical(unsigned occ, int nx, int ny, int nz) {
  if (nx > 0) occ = ((occ & 0x1249249u) << 2) | ((occ & 0x4924924u) >> 2) | (occ & 0x2492492u);
  if (ny > 0) occ = ((occ & 0x01c0e07u) << 6) | ((occ & 0x70381c0u) >> 6) | (occ & 0x0e07038u);
  if (nz > 0) occ = ((occ & 0x00001ffu) << 18) | ((occ & 0x7fc0000u) >> 18) | (occ & 0x003fe00u);
  return occ;
}

// G threads per edge (G = 1 for large batches: least work; G = 4 when few edges are in flight:
// shorter critical path): transform (A.1: double math, float store), exact 5-NN, line gate
// (centroid, scatter, eigenvalues in FP64) and the residual block {c, a, b, valid}.
template <int G>
__global__ void __launch_bounds__(kAssocThreads, G == 1 ? kAssocMinBlocks1 : 8) k_associate(DevBuffers d, int lane0, int outer_it, int force,
                                                                             const double* pose_override, int shard_rank, int shard_world) {
  const DevParams& p = d.p;
  const int lane_b = lane_at(d, lane0 + blockIdx.y);
  const OdomState& os = d.ostate[lane_b];
  const bool active = force || os.init;
  const int share = shard_world > 1 ? edge_share(os.n_edges, shard_world) : 0;
  const int E = shard_world > 1 ? min(os.n_edges, (shard_rank + 1) * share) : os.n_edges;
  const int t = shard_rank * share + (blockIdx.x * kAssocThreads + threadIdx.x) / G;
  const int ln = threadIdx.x & 31;
  const int gl = ln & (G - 1);                                   // lane inside the edge's group
  const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (ln & ~(G - 1)));
  if (active && (t - ln / G) < E) {   // warp-uniform: the fallback search below is cooperative
    const WinState& ws = d.wstate[lane_b];
    const double* T = pose_override ? pose_override : os.odom;
    const bool mine = t < E;
    // thread -> edge: Morton order from k_edge_order (identity on the stand-alone test path)
    const int e = (mine && !force) ? d.perm[(size_t)lane_b * p.Ecap + t] : t;
    const float4 c = mine ? d.edges[(size_t)lane_b * p.Ecap + e] : make_float4(0.f, 0.f, 0.f, 0.f);
    const float qx = xform_row(T, c.x, c.y, c.z), qy = xform_row(T + 4, c.x, c.y, c.z), qz = xform_row(T + 8, c.x, c.y, c.z);
    const unsigned gen = ws.gen & ((1u << kGenBits) - 1u);
    const unsigned hmask = (unsigned)p.Hcap - 1u, bmask = (unsigned)p.Bwords - 1u;
    const HashEntry* tab = d.htab + (size_t)lane_b * p.Hcap;
    const float4* sorted = d.sorted + (size_t)lane_b * p.Pcap;
    const unsigned* bloom = d.bloom + (size_t)lane_b * p.Bwords;
    Knn5 k;
#pragma unroll
    for (int r = 0; r < 5; ++r) k.k[r] = kEmptyCand;
    const bool searchable = mine && ws.hash_points > 0 && isfinite(qx) && isfinite(qy) && isfinite(qz);
    const int cx = cell_of(qx), cy = cell_of(qy), cz = cell_of(qz);
    // ---- level 1: the 27-cell cube, own cell first (it sets the pruning bound), then its 9 x-rows.
    // (A cell-major variant — the warp walking the union of its cubes with broadcast loads — and a
    // warp-per-edge variant with the buckets concatenated across the lanes were measured slower.)
    if (G == 1) {
      if (searchable) {
        // the 9 occupancy words of the cube are requested together with the own cell's probe (10 loads in
        // flight, one round trip) instead of one dependent load per row
        unsigned occ = 0;
#pragma unroll
        for (int r = 0; r < 9; ++r) occ |= bloom_row(bloom, bmask, cx - 1, 3, cy + r % 3 - 1, cz + r / 3 - 1) << (3 * r);
        const uint2 sc = hash_lookup(tab, hmask, gen, cx, cy, cz);
        knn_scan_bucket(sorted + sc.x, sc.y, qx, qy, qz, 3.0e38f, k);
        // neighbours nearest first (per axis: own, then the side of the nearer face, then the far side), so
        // that the bound tightens before the far cells are looked at and most of them fall to cell_min_d2
        const int nx = __fsub_rn(qx, kCell * (float)cx) < 0.5f * kCell ? -1 : 1;
        const int ny = __fsub_rn(qy, kCell * (float)cy) < 0.5f * kCell ? -1 : 1;
        const int nz = __fsub_rn(qz, kCell * (float)cz) < 0.5f * kCell ? -1 : 1;
        occ = occ_canonical(occ & ~(1u << 13), nx, ny, nz);
        for (int i = 1; i < 27 && occ; ++i) {
          const unsigned bit = kNearMask[i];
          if (!(occ & bit)) continue;
          occ &= ~bit;
          int dx, dy, dz;
          near_offsets(i, nx, ny, nz, &dx, &dy, &dz);
          knn_scan_cell(tab, sorted, hmask, gen, cx + dx, cy + dy, cz + dz, qx, qy, qz, 3.0e38f, k);
        }
      }
    } else {
      // the group strides over the own cell together, shares the tightest 5th-best as a bound, splits
      // the 9 rows round-robin and merges the G sorted lists by 5 rounds of group arg-min
      if (searchable) {
        const uint2 sc = hash_lookup(tab, hmask, gen, cx, cy, cz);
        for (unsigned j = gl; j < sc.y; j += G) knn_offer(__ldg(sorted + sc.x + j), qx, qy, qz, 3.0e38f, k);
      }
      const unsigned ubb = __reduce_min_sync(gmask, (unsigned)(k.k[4] >> 32));
      const float ub = __uint_as_float(ubb);   // 1.0 when the list is not full yet
      if (searchable)
        for (int r = gl; r < 9; r += G)
          knn_scan_row(tab, sorted, bloom, hmask, bmask, gen, cx - 1, 3, r == 4 ? 2u : 0u, cy + r % 3 - 1, cz + r / 3 - 1, qx, qy, qz, ub, k);
      __syncwarp(gmask);
      unsigned long long res[5];
#pragma unroll
      for (int r = 0; r < 5; ++r) {
        const unsigned hh = (unsigned)(k.k[0] >> 32), hl = (unsigned)k.k[0];
        const unsigned mh = __reduce_min_sync(gmask, hh);
        const unsigned ml = __reduce_min_sync(gmask, hh == mh ? hl : 0xffffffffu);
        const int wl = __ffs(__ballot_sync(gmask, hh == mh && hl == ml)) - 1;
        res[r] = ((unsigned long long)mh << 32) | ml;
        if (ln == wl) {
#pragma unroll
          for (int q = 0; q < 4; ++q) k.k[q] = k.k[q + 1];
          k.k[4] = kEmptyCand;
        }
      }
#pragma unroll
      for (int r = 0; r < 5; ++r) k.k[r] = res[r];   // the merged list, uniform over the group
    }
    knn_fallback_warp(tab, sorted, bloom, hmask, bmask, gen, searchable && gl == 0, qx, qy, qz, cx, cy, cz, k, ln);
    // G == 1 (large batches): the search ends here and the five neighbours go to k_line_gate, so that the search
    // kernel's register budget is not shared with the FP64 eigen-solver (no spills to speak of: -13 % at 128 lanes).
    // G > 1 (few edges in flight): gate in place — one launch less matters more there.
    bool match = false;
    if (mine && gl == 0) {
      int nn_idx[5];
#pragma unroll
      for (int r = 0; r < 5; ++r) nn_idx[r] = k.k[4] == kEmptyCand ? -1 : (int)(unsigned)k.k[r];
      if (G == 1) {
        int* nn_out = d.knn_out + ((size_t)lane_b * p.Ecap + e) * 5;
#pragma unroll
        for (int r = 0; r < 5; ++r) nn_out[r] = nn_idx[r];
      } else {
        match = line_gate(d, lane_b, e, c, nn_idx);
      }
      if (d.gate) knn_debug_out(d, lane_b, e, k, qx, qy, qz, c.w);
    }
    if (G != 1) {
      const int nm = __popc(__ballot_sync(0xffffffffu, match));
      if (ln == 0 && nm) atomicAdd(&d.diag[lane_b].n_matches[outer_it], nm);
    }
  }
  if (active && blockIdx.x == 0 && threadIdx.x == 0) d.diag[lane_b].n_map[outer_it] = d.wstate[lane_b].hash_points;
}

// ---------------------------------------------------------------------------------------
// Large batches: thread-per-edge set-up, candidates pooled over the warp (the default for the second outer iteration).
//
// Replay of the C1 data (tools/assoc_warp_sim.py): a warp of the thread-per-edge kernel spends 62 four-candidate
// iterations per 32 edges, 12 on the own cells and 50 on neighbour cells, although the 32 edges together hold only 16
// iterations' worth of candidates: neighbouring edges differ widely in how many neighbour points survive their bound.
// So the search is split:
//   phase A  one thread per edge.  An edge with a bound in hand LISTS (start, count) in shared memory every cell the
//            bound cannot exclude; an edge without one scans in place (own cell, then the neighbour cells nearest
//            first) until it holds five candidates, and lists the rest.  In the second outer iteration the bound is
//            there from the start — the largest distance to the five neighbours of the first iteration — so the own
//            cell is listed too and nothing is scanned in place;
//   phase B  the warp's listed buckets form one candidate sequence that is cut into 32 equal chunks; every lane scans
//            one chunk on behalf of the owning edges (query and bound read from shared memory) and splices the
//            candidates that pass the owner's bound (3 - 6 per edge) into the owner's list in a per-warp pool;
//   phase C  every owner merges its list into its five best.
// The candidate set an edge sees is a superset of the one the thread-per-edge kernel examines under its progressively
// tightened bound, every rejected candidate is beyond a bound the edge already holds, and the five best of a set do
// not depend on the order of insertion: results are bit-identical.  When the pool runs over, owners that lost a
// candidate scan their listed buckets themselves.
// ---------------------------------------------------------------------------------------
constexpr int kPoolSegs = 8;       // listed neighbour buckets per edge (further ones are scanned in place)
constexpr int kPoolSurv = 224;     // pooled candidates per warp that passed their owner's bound
constexpr unsigned kPoolNil = 0xffffu;

struct PoolWarp {
  uint2 seg[kPoolSegs][32];
  float qx[32], qy[32], qz[32], ub[32];
  unsigned pre[33];                       // exclusive prefix of the listed candidates per owner lane
  unsigned head[32];                      // owner's list of pooled candidates
  unsigned long long surv[kPoolSurv];
  unsigned short next[kPoolSurv];
  unsigned char nseg[32];
  unsigned nsurv, lost;                   // allocation counter; owners that lost a candidate to a full pool
};

__device__ __forceinline__ void knn_insert(unsigned long long key, Knn5& k) {
  if (key < k.k[4]) {
    knn_place(key, k.k);
  }
}

// d2 of a pooled candidate to its owner's query, and whether it passes the owner's bound
__device__ __forceinline__ bool pool_test(const float4& pt, float qx, float qy, float qz, float ub, unsigned long long* key) {
  const float ddx = __fsub_rn(qx, pt.x), ddy = __fsub_rn(qy, pt.y), ddz = __fsub_rn(qz, pt.z);
  const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(ddx, ddx), __fmul_rn(ddy, ddy)), __fmul_rn(ddz, ddz));
  *key = ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned)__float_as_int(pt.w);
  return d2 < 1.0f && d2 <= ub;
}

__global__ void __launch_bounds__(kAssocThreads, 16) k_associate_pool(DevBuffers d, int lane0, int outer_it, int force,
                                                                                  const double* pose_override, int shard_rank, int shard_world) {
  const DevParams& p = d.p;
  const int lane_b = lane_at(d, lane0 + blockIdx.y);
  const OdomState& os = d.ostate[lane_b];
  const bool active = force || os.init;
  const int share = shard_world > 1 ? edge_share(os.n_edges, shard_world) : 0;
  const int E = shard_world > 1 ? min(os.n_edges, (shard_rank + 1) * share) : os.n_edges;
  const int t = shard_rank * share + blockIdx.x * kAssocThreads + threadIdx.x;
  const int ln = threadIdx.x & 31;
  __shared__ PoolWarp smw[kAssocThreads / 32];
  if (active && (t - ln) < E) {   // warp-uniform
    PoolWarp& sm = smw[threadIdx.x >> 5];
    const WinState& ws = d.wstate[lane_b];
    const double* T = pose_override ? pose_override : os.odom;
    const bool mine = t < E;
    const int e = (mine && !force) ? d.perm[(size_t)lane_b * p.Ecap + t] : t;
    const float4 c = mine ? d.edges[(size_t)lane_b * p.Ecap + e] : make_float4(0.f, 0.f, 0.f, 0.f);
    const float qx = xform_row(T, c.x, c.y, c.z), qy = xform_row(T + 4, c.x, c.y, c.z), qz = xform_row(T + 8, c.x, c.y, c.z);
    const unsigned gen = ws.gen & ((1u << kGenBits) - 1u);
    const unsigned hmask = (unsigned)p.Hcap - 1u, bmask = (unsigned)p.Bwords - 1u;
    const HashEntry* tab = d.htab + (size_t)lane_b * p.Hcap;
    const float4* sorted = d.sorted + (size_t)lane_b * p.Pcap;
    const unsigned* bloom = d.bloom + (size_t)lane_b * p.Bwords;
    Knn5 k;
#pragma unroll
    for (int r = 0; r < 5; ++r) k.k[r] = kEmptyCand;
    const bool searchable = mine && ws.hash_points > 0 && isfinite(qx) && isfinite(qy) && isfinite(qz);
    const int cx = cell_of(qx), cy = cell_of(qy), cz = cell_of(qz);
    // ---- phase A
    int nseg = 0;
    unsigned listed = 0;
    // Second outer iteration (src/laser_odometry.cc:198): the map is the same as in the first and the pose moved by
    // millimetres, so the five neighbours found then (still in knn_out) are five map points close to this query and the
    // largest of their distances bounds the 5th-best distance from above.  With a bound in hand from the start nothing
    // is scanned in place: the own cell is listed like the others and the whole search runs pooled.
    float seed = 3.0e38f;
    if (searchable && outer_it == 1 && !force && shard_world == 1) {
      const int* prev = d.knn_out + ((size_t)lane_b * p.Ecap + e) * 5;
      if (prev[0] >= 0) {
        const float4* lin = d.lin + (size_t)lane_b * p.LinCap;
        const unsigned lmask = (unsigned)p.LinCap - 1u;
        float m = 0.0f;
#pragma unroll
        for (int r = 0; r < 5; ++r) {
          const float4 pt = lin[(unsigned)prev[r] & lmask];
          const float ddx = __fsub_rn(qx, pt.x), ddy = __fsub_rn(qy, pt.y), ddz = __fsub_rn(qz, pt.z);
          m = fmaxf(m, __fadd_rn(__fadd_rn(__fmul_rn(ddx, ddx), __fmul_rn(ddy, ddy)), __fmul_rn(ddz, ddz)));
        }
        if (m == m) seed = m;   // not NaN
      }
    }
    const bool seeded = seed < 3.0e38f;
    if (searchable) {
      unsigned occ = 0;
#pragma unroll
      for (int r = 0; r < 9; ++r) occ |= bloom_row(bloom, bmask, cx - 1, 3, cy + r % 3 - 1, cz + r / 3 - 1) << (3 * r);
      const uint2 own = hash_lookup(tab, hmask, gen, cx, cy, cz);   // in flight together with the occupancy words
      const int nx = __fsub_rn(qx, kCell * (float)cx) < 0.5f * kCell ? -1 : 1;
      const int ny = __fsub_rn(qy, kCell * (float)cy) < 0.5f * kCell ? -1 : 1;
      const int nz = __fsub_rn(qz, kCell * (float)cz) < 0.5f * kCell ? -1 : 1;
      occ = occ_canonical(occ | (1u << 13), nx, ny, nz);
      for (int i = 0; i < 27 && occ; ++i) {   // slot 0 = the own cell: one scan site for all in-place scans (code size)
        const unsigned bit = kNearMask[i];
        if (!(occ & bit)) continue;
        occ &= ~bit;
        int dx, dy, dz;
        near_offsets(i, nx, ny, nz, &dx, &dy, &dz);
        uint2 sc = own;
        if (i > 0) {
          const float dmin = cell_min_d2(qx, qy, qz, cx + dx, cy + dy, cz + dz);
          if (__float_as_uint(dmin) > (unsigned)(k.k[4] >> 32) || dmin > seed) continue;
          sc = hash_lookup(tab, hmask, gen, cx + dx, cy + dy, cz + dz);
        }
        if (sc.y == 0u) continue;
        if ((k.k[4] == kEmptyCand && !seeded) || nseg == kPoolSegs) {
          knn_scan_bucket(sorted + sc.x, sc.y, qx, qy, qz, seed, k);   // no bound yet (or list full)
        } else {
          sm.seg[nseg][ln] = sc; ++nseg; listed += sc.y;
        }
      }
    }
    // ---- phase B
    sm.qx[ln] = qx; sm.qy[ln] = qy; sm.qz[ln] = qz;
    // listed > 0 only with a bound in hand: five candidates, or the seed
    sm.ub[ln] = k.k[4] == kEmptyCand ? seed : fminf(seed, __uint_as_float((unsigned)(k.k[4] >> 32)));
    sm.nseg[ln] = (unsigned char)nseg;
    sm.head[ln] = kPoolNil;
    unsigned incl = listed;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned v = __shfl_up_sync(0xffffffffu, incl, o); if (ln >= o) incl += v; }
    sm.pre[ln + 1] = incl;
    if (ln == 0) { sm.pre[0] = 0u; sm.nsurv = 0u; sm.lost = 0u; }
    __syncwarp();
    const unsigned total = sm.pre[32];
    if (total) {   // warp-uniform
      const unsigned per = (total + 31u) >> 5;
      const unsigned pos = (unsigned)ln * per;
      unsigned rem = pos < total ? min(per, total - pos) : 0u;
      if (rem) {
        int o = 0;   // the owner whose listed range holds `pos`: the largest o with pre[o] <= pos
#pragma unroll
        for (int step = 16; step; step >>= 1) if (sm.pre[o + step] <= pos) o += step;
        unsigned off = pos - sm.pre[o];
        int s = 0;
        uint2 sg = sm.seg[0][o];
        while (off >= sg.y) { off -= sg.y; ++s; sg = sm.seg[s][o]; }
        unsigned j = sg.x + off, jend = sg.x + sg.y;
        float ox = sm.qx[o], oy = sm.qy[o], oz = sm.qz[o], oub = sm.ub[o];
        int ons = sm.nseg[o];
        while (rem) {
          if (j == jend) {   // next listed bucket of this owner, else of the next owner that listed any
            if (++s == ons) {
              do { ++o; ons = sm.nseg[o]; } while (ons == 0);
              s = 0; ox = sm.qx[o]; oy = sm.qy[o]; oz = sm.qz[o]; oub = sm.ub[o];
            }
            sg = sm.seg[s][o]; j = sg.x; jend = sg.x + sg.y;
          }
          const unsigned n = min(min(jend - j, rem), 4u), last = j + n - 1u;
          const float4 p0 = __ldg(sorted + j), p1 = __ldg(sorted + min(j + 1u, last));
          const float4 p2 = __ldg(sorted + min(j + 2u, last)), p3 = __ldg(sorted + min(j + 3u, last));
          unsigned long long key[4];
          bool ok[4];
          ok[0] = pool_test(p0, ox, oy, oz, oub, &key[0]);
          ok[1] = pool_test(p1, ox, oy, oz, oub, &key[1]) && n > 1u;
          ok[2] = pool_test(p2, ox, oy, oz, oub, &key[2]) && n > 2u;
          ok[3] = pool_test(p3, ox, oy, oz, oub, &key[3]) && n > 3u;
          const unsigned cnt = (unsigned)ok[0] + (unsigned)ok[1] + (unsigned)ok[2] + (unsigned)ok[3];
          if (cnt) {   // one allocation and one list splice for the (up to four) candidates of this owner
            const unsigned base = atomicAdd(&sm.nsurv, cnt);
            if (base + cnt <= (unsigned)kPoolSurv) {
              unsigned slot = base;
#pragma unroll
              for (int r = 0; r < 4; ++r)
                if (ok[r]) { sm.surv[slot] = key[r]; if (slot != base) sm.next[slot] = (unsigned short)(slot - 1u); ++slot; }
              sm.next[base] = (unsigned short)atomicExch(&sm.head[o], base + cnt - 1u);
            } else {
              atomicOr(&sm.lost, 1u << o);
            }
          }
          j += n; rem -= n;
        }
      }
      __syncwarp();
      // ---- phase C
      if ((sm.lost >> ln) & 1u) {
        for (int s = 0; s < nseg; ++s) {   // rare (a few % of the warps): a plain loop keeps the code small
          const uint2 sg = sm.seg[s][ln];
          for (unsigned j = 0; j < sg.y; ++j) knn_offer(__ldg(sorted + sg.x + j), qx, qy, qz, 3.0e38f, k);
        }
      } else {
        for (unsigned sl = sm.head[ln]; sl != kPoolNil; sl = sm.next[sl]) knn_insert(sm.surv[sl], k);
      }
      __syncwarp();
    }
    knn_fallback_warp(tab, sorted, bloom, hmask, bmask, gen, searchable, qx, qy, qz, cx, cy, cz, k, ln);
    if (mine) {
      int* nn_out = d.knn_out + ((size_t)lane_b * p.Ecap + e) * 5;
#pragma unroll
      for (int r = 0; r < 5; ++r) nn_out[r] = k.k[4] == kEmptyCand ? -1 : (int)(unsigned)k.k[r];
      if (d.gate) knn_debug_out(d, lane_b, e, k, qx, qy, qz, c.w);
    }
  }
  if (active && blockIdx.x == 0 && threadIdx.x == 0) d.diag[lane_b].n_map[outer_it] = d.wstate[lane_b].hash_points;
}

// The gate of every edge after a G == 1 search, one thread per edge in edge order (the edge-sharded mode: this
// rank's Morton positions).
__global__ void __launch_bounds__(128) k_line_gate(DevBuffers d, int lane0, int outer_it, int force, int shard_rank, int shard_world) {
  const DevParams& p = d.p;
  const int lane_b = lane_at(d, lane0 + blockIdx.y);
  const OdomState& os = d.ostate[lane_b];
  const bool active = force || os.init;
  const int share = shard_world > 1 ? edge_share(os.n_edges, shard_world) : 0;
  const int E = shard_world > 1 ? min(os.n_edges, (shard_rank + 1) * share) : os.n_edges;
  const int t = shard_rank * share + blockIdx.x * blockDim.x + threadIdx.x;
  bool match = false;
  if (active && t < E) {
    const int e = shard_world > 1 ? d.perm[(size_t)lane_b * p.Ecap + t] : t;   // unsharded: edge order (coalesced)
    const int* nn_in = d.knn_out + ((size_t)lane_b * p.Ecap + e) * 5;
    int nn_idx[5];
#pragma unroll
    for (int r = 0; r < 5; ++r) nn_idx[r] = nn_in[r];
    match = line_gate(d, lane_b, e, d.edges[(size_t)lane_b * p.Ecap + e], nn_idx);
  }
  const int nm = __popc(__ballot_sync(0xffffffffu, match));
  if ((threadIdx.x & 31) == 0 && nm) atomicAdd(&d.diag[lane_b].n_matches[outer_it], nm);
}
#undef MUL
#undef ADD
#undef SUB
#undef DIV

// Threads per edge: 1 for large batches (least total work); 4, 8 or 16 while the launch would otherwise leave most
// of the 148 SMs idle (shorter per-edge chains; measured per lane count).  Edge-sharded mode (world > 1): a rank's
// share is one partial wave, so the stage lasts as long as the longest per-edge chain; the idle threads go to shorter
// chains (the batched thresholds were measured on whole C1 batches).  LIODOM_ASSOC_GROUP=1|4|8|16 forces a variant
// (the parity tests cover all four).
// (The variant switches are read per launch — a getenv is ~100 ns against launches of 100+ us — so that one process,
// e.g. the parity tests, can run every variant.)
static int assoc_group_size(int edges_per_lane, int nlanes, int world) {
  if (const char* e = getenv("LIODOM_ASSOC_GROUP")) { const int v = atoi(e); if (v == 1 || v == 4 || v == 8 || v == 16) return v; }
  if (world > 1) return edges_per_lane <= 16384 ? 16 : (edges_per_lane <= 32768 ? 8 : 4);
  const long long edges_in_flight = (long long)edges_per_lane * nlanes;
  if (edges_in_flight <= 5632) return 16;
  if (edges_in_flight <= 2 * 5632) return 8;
  return edges_in_flight <= 12 * 5632 ? 4 : 1;
}

static void launch_associate_any(const DevBuffers& d, cudaStream_t s, int lane0, int nlanes, int edges_per_lane, int outer_it, int force,
                                 const double* pose_override, int rank, int world) {
  const int G = assoc_group_size(edges_per_lane, nlanes, world);
  const dim3 g((unsigned)(((long long)edges_per_lane * G + kAssocThreads - 1) / kAssocThreads), nlanes);
  if (G == 16) k_associate<16><<<g, kAssocThreads, 0, s>>>(d, lane0, outer_it, force, pose_override, rank, world);
  else if (G == 8) k_associate<8><<<g, kAssocThreads, 0, s>>>(d, lane0, outer_it, force, pose_override, rank, world);
  else if (G == 4) k_associate<4><<<g, kAssocThreads, 0, s>>>(d, lane0, outer_it, force, pose_override, rank, world);
  else {
    // The warp-pooled kernel is used where it wins: the second outer iteration, whose bound is seeded from the first
    // one's neighbours so that the whole search runs pooled (ncu at 128 lanes: 382 vs 446 us, 19 vs 11 active threads;
    // unseeded it is 463 vs 441 us — 64 registers and 10 KB of shared memory per CTA cost occupancy;
    // profiles/k_associate_pool_r02q_lanes128.txt).  LIODOM_ASSOC_POOL=0 / 1 forces never / always.
    const char* pool_env = getenv("LIODOM_ASSOC_POOL");
    const bool pooled = pool_env ? atoi(pool_env) == 1 : (outer_it == 1 && !force && world == 1);
    if (pooled) k_associate_pool<<<g, kAssocThreads, 0, s>>>(d, lane0, outer_it, force, pose_override, rank, world);
    else k_associate<1><<<g, kAssocThreads, 0, s>>>(d, lane0, outer_it, force, pose_override, rank, world);
    k_line_gate<<<dim3((edges_per_lane + 127) / 128, nlanes), 128, 0, s>>>(d, lane0, outer_it, force, rank, world);
  }
}

int launch_associate(const DevBuffers& d, cudaStream_t s, LaneRange lr, int outer_it, bool force, const double* pose_override) {
  launch_associate_any(d, s, lr.lane0, lr.nlanes, d.p.Ecap, outer_it, force ? 1 : 0, pose_override, 0, 1);
  return 2;
}
int launch_associate_shard(const DevBuffers& d, cudaStream_t s, int lane, int outer_it, int rank, int world) {
  launch_associate_any(d, s, lane, 1, edge_share(d.p.Ecap, world), outer_it, 0, nullptr, rank, world);
  return 2;
}

// ---------------------------------------------------------------------------------------
// window update (src/laser_odometry.cc:231-235 and the first-frame branch :121-136)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_window_update(DevBuffers d, int lane0) {
  const DevParams& p = d.p;
  const int lane_b = lane_at(d, lane0 + blockIdx.x);
  OdomState& os = d.ostate[lane_b];
  WinState& ws = d.wstate[lane_b];
  const int E = os.n_edges;
  const int s = (ws.head + ws.nframes) % p.slots;
  float4* slab = d.win + ((size_t)lane_b * p.slots + s) * p.Ecap;
  const float4* edges = d.edges + (size_t)lane_b * p.Ecap;
  const bool init = os.init != 0;
  for (int i = threadIdx.x; i < E; i += blockDim.x) {
    const float4 c = edges[i];
    if (!init) slab[i] = c;  // first frame: lmap_manager.addPointCloud(feats) untouched
    else {
      const double* T = os.odom;
      slab[i] = make_float4(__double2float_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(T[0], c.x), __dmul_rn(T[1], c.y)), __dmul_rn(T[2], c.z)), T[3])),
                            __double2float_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(T[4], c.x), __dmul_rn(T[5], c.y)), __dmul_rn(T[6], c.z)), T[7])),
                            __double2float_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(T[8], c.x), __dmul_rn(T[9], c.y)), __dmul_rn(T[10], c.z)), T[11])),
                            c.w);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const int lane_c = lane_at(d, lane0 + blockIdx.x);   // looked up again: keeping lane_b across the barrier spills
    OdomState& os_c = d.ostate[lane_c];
    win_commit(d, lane_c, E);
    hash_begin(d, lane_c);
    os_c.init = 1; os_c.frame++;
    double* po = d.poses_out + (size_t)lane_c * 16;
    for (int k = 0; k < 12; ++k) po[k] = os_c.odom[k];
    po[12] = po[13] = po[14] = 0.0; po[15] = 1.0;
  }
}

int launch_window_update(const DevBuffers& d, cudaStream_t s, LaneRange lr) {
  k_window_update<<<lr.nlanes, 1024, 0, s>>>(d, lr.lane0);
  return 1 + launch_hash_build(d, s, lr);
}

// LocalMapManager::addPointCloud from a device staging buffer (API / tests).
__global__ void __launch_bounds__(1024) k_lmap_add(DevBuffers d, int lane_b, const float4* pts, int n) {
  const DevParams& p = d.p;
  WinState& ws = d.wstate[lane_b];
  const int s = (ws.head + ws.nframes) % p.slots;
  float4* slab = d.win + ((size_t)lane_b * p.slots + s) * p.Ecap;
  for (int i = threadIdx.x; i < n; i += blockDim.x) slab[i] = pts[i];
  __syncthreads();
  if (threadIdx.x == 0) { win_commit(d, lane_b, n); hash_begin(d, lane_b); }
}

int launch_lmap_add(const DevBuffers& d, cudaStream_t s, int lane, const float4* pts_dev, int n) {
  k_lmap_add<<<1, 1024, 0, s>>>(d, lane, pts_dev, n);
  return 1 + launch_hash_build(d, s, LaneRange{lane, 1});
}

// rebuild the hash of one lane after the window / received map was edited from the host
__global__ void k_hash_begin(DevBuffers d, int lane_b) { if (threadIdx.x == 0) hash_begin(d, lane_b, true); }
int launch_hash_rebuild(const DevBuffers& d, cudaStream_t s, int lane) {
  k_hash_begin<<<1, 32, 0, s>>>(d, lane);
  return 1 + launch_hash_build(d, s, LaneRange{lane, 1});
}

// gather the window in logical order (LocalMapManager::getLocalMap)
__global__ void __launch_bounds__(256) k_lmap_gather(DevBuffers d, int lane_b, float4* out) {
  WinView v;
  load_win_view(d, lane_b, &v, false);   // LocalMapManager::getLocalMap returns the unfiltered window
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < v.total; i += gridDim.x * blockDim.x) out[i] = win_point(d, lane_b, v, i);
}
int launch_lmap_gather(const DevBuffers& d, cudaStream_t s, int lane, float4* out) {
  k_lmap_gather<<<64, 256, 0, s>>>(d, lane, out);
  return 1;
}

}  // namespace liodom
