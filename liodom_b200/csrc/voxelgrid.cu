// filter_local_map on sm_100a: pcl::VoxelGrid(leaf 0.4) of the sliding window as the kNN target
// (replaces LaserOdometer::computeLocalMap, src/laser_odometry.cc:274-298, filter branch :286-292).
//
// pcl::VoxelGrid<PointXYZI>::applyFilter semantics kept (SURVEY.md App. A.3):
//   inverse leaf = 1 / 0.4f in float; bounding box of the finite points; min_b = floor(min * inv),
//   div_b = floor(max * inv) - min_b + 1; voxel index of a point = i + j * div_x + k * div_x * div_y
//   with i = int(floor(x * inv) - float(min_b.x)) (float math); one output point per occupied voxel
//   in ascending index order = centroid of x, y, z and intensity, float sums accumulated in input
//   order then divided by the count.  If the index space exceeds int32 PCL warns and returns the
//   input unchanged: the filter then stays off for that build.
//
// Mapping: every lane of the batch is filtered by the same launches, grid (tiles, lanes).
//   bbox (atomic min/max on order-preserving integer images of the floats) -> plan (one thread per
//   lane) -> voxel index per point -> stable LSD radix sort of (index, logical position), 8-bit
//   digits, only as many passes as the index range needs -> voxel heads per tile -> one thread per
//   voxel walks its (input-ordered) run and writes the centroid at the voxel's rank.
// The file is compiled with -fmad=false; the float operations below are the reference's, one rounding each.
#include "common.cuh"

namespace liodom {

constexpr float kVgLeaf = 0.4f;                  // src/laser_odometry.cc:290

__device__ __forceinline__ unsigned f2ord(float f) { const unsigned b = __float_as_uint(f); return (b & 0x80000000u) ? ~b : (b | 0x80000000u); }
__device__ __forceinline__ float ord2f(unsigned o) { return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o); }
__device__ __forceinline__ bool finite3(const float4& p) { return isfinite(p.x) && isfinite(p.y) && isfinite(p.z); }

// Lanes whose window is not filtered in this build leave every kernel at once.
#define VG_LANE_PROLOGUE                                   \
  const int lane_b = lane_at(d, lane0 + blockIdx.y);       \
  WinState& ws = d.wstate[lane_b];                         \
  if (!ws.vg_active) return;                               \
  const int n = ws.view_prefix[ws.nframes];                \
  const int tile0 = blockIdx.x * kVgTile;                  \
  if (tile0 >= n && blockIdx.x != 0) return;

__global__ void __launch_bounds__(256) k_vg_bbox(DevBuffers d, int lane0) {
  VG_LANE_PROLOGUE
  WinView v;
  load_win_view(d, lane_b, &v, false);
  unsigned lo[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, hi[3] = {0u, 0u, 0u};
  for (int k = threadIdx.x; k < kVgTile; k += 256) {
    const int i = tile0 + k;
    if (i >= n) break;
    const float4 p = win_point(d, lane_b, v, i);
    if (!finite3(p)) continue;
    const unsigned ex = f2ord(p.x), ey = f2ord(p.y), ez = f2ord(p.z);
    lo[0] = min(lo[0], ex); lo[1] = min(lo[1], ey); lo[2] = min(lo[2], ez);
    hi[0] = max(hi[0], ex); hi[1] = max(hi[1], ey); hi[2] = max(hi[2], ez);
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    lo[a] = __reduce_min_sync(0xffffffffu, lo[a]);
    hi[a] = __reduce_max_sync(0xffffffffu, hi[a]);
  }
  if ((threadIdx.x & 31) == 0)
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      if (lo[a] != 0xffffffffu) atomicMin(&ws.vg_lo[a], lo[a]);
      if (hi[a] != 0u) atomicMax(&ws.vg_hi[a], hi[a]);
    }
}

// One thread per lane: min_b / div_b, the int32 overflow rule and the number of radix passes.
__global__ void k_vg_plan(DevBuffers d, int lane0, int nlanes) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= nlanes) return;
  WinState& ws = d.wstate[lane_at(d, lane0 + l)];
  if (!ws.vg_active) return;
  if (ws.vg_lo[0] == 0xffffffffu) {   // no finite point: the filtered cloud is empty
    ws.vg_passes = 0; ws.vg_div[0] = ws.vg_div[1] = ws.vg_div[2] = 0; ws.vg_invalid = 0u;
    return;
  }
  const float inv = __fdiv_rn(1.0f, kVgLeaf);
  long long dd[3];
  for (int a = 0; a < 3; ++a) {
    const float mn = ord2f(ws.vg_lo[a]), mx = ord2f(ws.vg_hi[a]);
    dd[a] = (long long)__fmul_rn(__fsub_rn(mx, mn), inv) + 1;
    ws.vg_minb[a] = (int)floorf(__fmul_rn(mn, inv));
    ws.vg_div[a] = (int)floorf(__fmul_rn(mx, inv)) - ws.vg_minb[a] + 1;
  }
  if (dd[0] * dd[1] * dd[2] > 2147483647ll) { ws.vg_active = 0; return; }   // PCL: "leaf size too small", input returned unchanged
  const long long cells = (long long)ws.vg_div[0] * ws.vg_div[1] * ws.vg_div[2];
  if (cells > 2147483646ll) { ws.vg_active = 0; return; }
  // non-finite points get the key `cells` (above every voxel index, so they sort last and form no voxel)
  ws.vg_invalid = (unsigned)cells;
  int bits = 1;
  while ((1ll << bits) <= cells) ++bits;
  ws.vg_passes = (bits + 7) / 8;
}

__global__ void __launch_bounds__(256) k_vg_keys(DevBuffers d, int lane0) {
  VG_LANE_PROLOGUE
  WinView v;
  load_win_view(d, lane_b, &v, false);
  const float inv = __fdiv_rn(1.0f, kVgLeaf);
  const float bx = (float)ws.vg_minb[0], by = (float)ws.vg_minb[1], bz = (float)ws.vg_minb[2];
  const int mul1 = ws.vg_div[0], mul2 = ws.vg_div[0] * ws.vg_div[1];
  unsigned* key = d.vg_key[0] + (size_t)lane_b * d.p.Wcap;
  unsigned* val = d.vg_val[0] + (size_t)lane_b * d.p.Wcap;
  for (int k = threadIdx.x; k < kVgTile; k += 256) {
    const int i = tile0 + k;
    if (i >= n) break;
    const float4 p = win_point(d, lane_b, v, i);
    unsigned idx = ws.vg_invalid;
    if (finite3(p)) {
      const int i0 = (int)__fsub_rn(floorf(__fmul_rn(p.x, inv)), bx);
      const int i1 = (int)__fsub_rn(floorf(__fmul_rn(p.y, inv)), by);
      const int i2 = (int)__fsub_rn(floorf(__fmul_rn(p.z, inv)), bz);
      idx = (unsigned)(i0 + i1 * mul1 + i2 * mul2);
    }
    key[i] = idx; val[i] = (unsigned)i;
  }
}

// ---- stable LSD radix sort, 8-bit digits, every lane in the same launch ---------------------------
__global__ void __launch_bounds__(256) k_vg_hist(DevBuffers d, int lane0, int pass) {
  VG_LANE_PROLOGUE
  if (pass >= ws.vg_passes) return;
  __shared__ int h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const unsigned* key = d.vg_key[pass & 1] + (size_t)lane_b * d.p.Wcap;
  const int shift = pass * 8;
  for (int k = threadIdx.x; k < kVgTile; k += 256) {
    const int i = tile0 + k;
    if (i < n) atomicAdd(&h[(key[i] >> shift) & 255u], 1);
  }
  __syncthreads();
  d.vg_hist[(size_t)lane_b * 256 * d.p.vg_blocks + (size_t)threadIdx.x * d.p.vg_blocks + blockIdx.x] = h[threadIdx.x];
}

// exclusive scan of the lane's digit-major histogram (256 * tiles entries) by one CTA
__global__ void __launch_bounds__(1024) k_vg_scan(DevBuffers d, int lane0, int pass) {
  const int lane_b = lane_at(d, lane0 + blockIdx.x);
  const WinState& ws = d.wstate[lane_b];
  if (!ws.vg_active || pass >= ws.vg_passes) return;
  const int n = ws.view_prefix[ws.nframes];
  const int tiles = (n + kVgTile - 1) / kVgTile, nb = d.p.vg_blocks;
  int* hist = d.vg_hist + (size_t)lane_b * 256 * nb;
  __shared__ int s[1024];
  __shared__ int carry;
  const int tid = threadIdx.x;
  if (tid == 0) carry = 0;
  __syncthreads();
  // logical sequence: digit-major over the used tiles only (entry e -> digit e / tiles, tile e % tiles)
  const int m = 256 * tiles;
  for (int base = 0; base < m; base += 4096) {
    int vv[4], sum = 0;
    for (int k = 0; k < 4; ++k) {
      const int e = base + tid * 4 + k;
      vv[k] = e < m ? hist[(e / tiles) * nb + (e % tiles)] : 0;
      sum += vv[k];
    }
    s[tid] = sum;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
      const int t = tid >= o ? s[tid - o] : 0;
      __syncthreads();
      s[tid] += t;
      __syncthreads();
    }
    int run = carry + s[tid] - sum;
    for (int k = 0; k < 4; ++k) {
      const int e = base + tid * 4 + k;
      if (e < m) hist[(e / tiles) * nb + (e % tiles)] = run;
      run += vv[k];
    }
    __syncthreads();
    if (tid == 1023) carry += s[1023];
    __syncthreads();
  }
}

// stable scatter: each warp owns a contiguous 256-key run of the tile, processed in 8 rounds of 32
__global__ void __launch_bounds__(256) k_vg_scatter(DevBuffers d, int lane0, int pass) {
  VG_LANE_PROLOGUE
  if (pass >= ws.vg_passes) return;
  __shared__ int wcnt[8][256];
  for (int k = threadIdx.x; k < 8 * 256; k += 256) (&wcnt[0][0])[k] = 0;
  __syncthreads();
  const size_t lo = (size_t)lane_b * d.p.Wcap;
  const unsigned* kin = d.vg_key[pass & 1] + lo;
  const unsigned* vin = d.vg_val[pass & 1] + lo;
  unsigned* kout = d.vg_key[(pass & 1) ^ 1] + lo;
  unsigned* vout = d.vg_val[(pass & 1) ^ 1] + lo;
  const int shift = pass * 8;
  const int w = threadIdx.x >> 5, ln = threadIdx.x & 31;
  int dg[8];
  unsigned kk[8];
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int i = tile0 + w * 256 + r * 32 + ln;
    kk[r] = i < n ? kin[i] : 0u;
    const int dgt = i < n ? (int)((kk[r] >> shift) & 255u) : -1;
    dg[r] = dgt;
    const unsigned mm = __match_any_sync(0xffffffffu, dgt);
    if (dgt >= 0 && (__ffs(mm) - 1) == ln) wcnt[w][dgt] += __popc(mm);
    __syncwarp();
  }
  __syncthreads();
  {
    const int dgt = threadIdx.x;
    int run = d.vg_hist[(size_t)lane_b * 256 * d.p.vg_blocks + (size_t)dgt * d.p.vg_blocks + blockIdx.x];
#pragma unroll
    for (int ww = 0; ww < 8; ++ww) { const int c = wcnt[ww][dgt]; wcnt[ww][dgt] = run; run += c; }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int i = tile0 + w * 256 + r * 32 + ln;
    const int dgt = dg[r];
    const unsigned mm = __match_any_sync(0xffffffffu, dgt);
    if (dgt >= 0) {
      const int pos = wcnt[w][dgt] + __popc(mm & ((1u << ln) - 1u));
      kout[pos] = kk[r]; vout[pos] = vin[i];
    }
    __syncwarp();
    if (dgt >= 0 && (__ffs(mm) - 1) == ln) wcnt[w][dgt] += __popc(mm);
    __syncwarp();
  }
}

// voxels (runs of equal keys) starting in each tile
__global__ void __launch_bounds__(256) k_vg_heads(DevBuffers d, int lane0) {
  VG_LANE_PROLOGUE
  const unsigned* key = d.vg_key[ws.vg_passes & 1] + (size_t)lane_b * d.p.Wcap;
  const unsigned kVgInvalid = ws.vg_invalid;
  int c = 0;
  for (int k = threadIdx.x; k < kVgTile; k += 256) {
    const int i = tile0 + k;
    if (i < n) { const unsigned kk = key[i]; c += (kk != kVgInvalid && (i == 0 || key[i - 1] != kk)) ? 1 : 0; }
  }
  __shared__ int s[8];
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) { int t = 0; for (int k = 0; k < 8; ++k) t += s[k]; d.vg_heads[(size_t)lane_b * d.p.vg_blocks + blockIdx.x] = t; }
}

// centroid of every voxel, written at the voxel's rank; the lane's target size becomes the voxel count
__global__ void __launch_bounds__(256) k_vg_emit(DevBuffers d, int lane0) {
  VG_LANE_PROLOGUE
  const int tiles = (n + kVgTile - 1) / kVgTile;
  const int* heads = d.vg_heads + (size_t)lane_b * d.p.vg_blocks;
  __shared__ int s_warp[8];
  __shared__ int s_base, s_total;
  {   // voxels before this tile (and, in tile 0, the lane's total)
    int before = 0, total = 0;
    for (int k = threadIdx.x; k < tiles; k += 256) { const int h = heads[k]; total += h; if (k < (int)blockIdx.x) before += h; }
    for (int o = 16; o > 0; o >>= 1) { before += __shfl_xor_sync(0xffffffffu, before, o); total += __shfl_xor_sync(0xffffffffu, total, o); }
    __shared__ int sb[8], st[8];
    if ((threadIdx.x & 31) == 0) { sb[threadIdx.x >> 5] = before; st[threadIdx.x >> 5] = total; }
    __syncthreads();
    if (threadIdx.x == 0) {
      int b = 0, t = 0;
      for (int k = 0; k < 8; ++k) { b += sb[k]; t += st[k]; }
      s_base = b; s_total = t;
    }
    __syncthreads();
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) ws.hash_points = tiles > 0 ? s_total : 0;
  if (tile0 >= n) return;
  WinView v;
  load_win_view(d, lane_b, &v, false);
  const size_t lo = (size_t)lane_b * d.p.Wcap;
  const unsigned* key = d.vg_key[ws.vg_passes & 1] + lo;
  const unsigned* val = d.vg_val[ws.vg_passes & 1] + lo;
  float4* out = d.filtered + lo;
  const unsigned kVgInvalid = ws.vg_invalid;
  // thread t owns the 8 consecutive keys tile0 + 8 t .. + 7: head flags, then a block-wide exclusive scan
  const int first = tile0 + threadIdx.x * 8;
  unsigned flags = 0;
  unsigned prev = (first > 0 && first <= n) ? key[first - 1] : 0xffffffffu;
  unsigned kk[8];
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int i = first + r;
    kk[r] = i < n ? key[i] : kVgInvalid;
    if (kk[r] != kVgInvalid && (i == 0 || kk[r] != prev)) flags |= 1u << r;
    prev = kk[r];
  }
  const int mine = __popc(flags);
  int incl = mine;
  const int ln = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (ln >= o) incl += t; }
  if (ln == 31) s_warp[w] = incl;
  __syncthreads();
  int wbase = 0;
  for (int k = 0; k < w; ++k) wbase += s_warp[k];
  int rank = s_base + wbase + incl - mine;
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    if (!(flags & (1u << r))) continue;
    const unsigned k0 = kk[r];
    float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
    int cnt = 0;
    for (int u = first + r; u < n && key[u] == k0; ++u) {   // pcl::CentroidPoint, input order
      const float4 p = win_point(d, lane_b, v, (int)val[u]);
      sx = __fadd_rn(sx, p.x); sy = __fadd_rn(sy, p.y); sz = __fadd_rn(sz, p.z); si = __fadd_rn(si, p.w);
      ++cnt;
    }
    const float fc = (float)cnt;
    out[rank++] = make_float4(__fdiv_rn(sx, fc), __fdiv_rn(sy, fc), __fdiv_rn(sz, fc), __fdiv_rn(si, fc));
  }
}
#undef VG_LANE_PROLOGUE

int launch_window_filter(const DevBuffers& d, cudaStream_t s, LaneRange lr) {
  if (!d.filtered || !d.p.filter_local_map || d.p.mapping || d.p.vg_blocks <= 0) return 0;
  const dim3 g(d.p.vg_blocks, lr.nlanes);
  int k = 0;
  k_vg_bbox<<<g, 256, 0, s>>>(d, lr.lane0); ++k;
  k_vg_plan<<<(lr.nlanes + 63) / 64, 64, 0, s>>>(d, lr.lane0, lr.nlanes); ++k;
  k_vg_keys<<<g, 256, 0, s>>>(d, lr.lane0); ++k;
  for (int pass = 0; pass < 4; ++pass) {
    k_vg_hist<<<g, 256, 0, s>>>(d, lr.lane0, pass);
    k_vg_scan<<<lr.nlanes, 1024, 0, s>>>(d, lr.lane0, pass);
    k_vg_scatter<<<g, 256, 0, s>>>(d, lr.lane0, pass);
    k += 3;
  }
  k_vg_heads<<<g, 256, 0, s>>>(d, lr.lane0); ++k;
  k_vg_emit<<<g, 256, 0, s>>>(d, lr.lane0); ++k;
  return k;
}

}  // namespace liodom
