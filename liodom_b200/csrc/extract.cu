// FeatureExtractor hot path on sm_100a: ring split, 11-tap curvature, per-region greedy
// top-k with +-5 suppression (replaces src/feature_extractor.cc:84-313 of the reference).
//
// Compiled with -fmad=false; the float/double sequences below additionally use the
// explicit round-to-nearest intrinsics so that no contraction can change a rounding
// (the reference is built without -march, i.e. SSE2 without FMA, CMakeLists.txt:13).
#include "common.cuh"
#include <math_constants.h>
#include <cstdlib>

namespace liodom {

// ---------------------------------------------------------------------------------------
// A1 + A2: isValidPoint + ring id (src/feature_extractor.cc:84-102, :126-151, :160-175)
// ---------------------------------------------------------------------------------------
// FLOAT32 field at an arbitrary byte address (PointCloud2 point_step need not be a multiple of 4,
// e.g. the 22-byte velodyne PointXYZIRT): little-endian bytes, as pcl::fromROSMsg's memcpy reads them.
__device__ __forceinline__ float load_f32_bytes(const char* p) {
  if ((reinterpret_cast<uintptr_t>(p) & 3) == 0) return __ldg(reinterpret_cast<const float*>(p));
  const unsigned char* b = reinterpret_cast<const unsigned char*>(p);
  return __uint_as_float((unsigned)__ldg(b) | ((unsigned)__ldg(b + 1) << 8) | ((unsigned)__ldg(b + 2) << 16) | ((unsigned)__ldg(b + 3) << 24));
}
__device__ __forceinline__ const char* point_base(const ScanDesc& sc, int i) {
  const char* base = reinterpret_cast<const char*>(sc.pts);
  if (sc.generic && sc.row_step) return base + (size_t)(i / sc.width) * sc.row_step + (size_t)(i % sc.width) * sc.stride_bytes;
  return base + (size_t)i * sc.stride_bytes;
}
__device__ __forceinline__ void load_xyz(const ScanDesc& sc, int i, float& x, float& y, float& z) {
  const char* base = point_base(sc, i);
  if (sc.generic) {
    x = load_f32_bytes(base + sc.off_x); y = load_f32_bytes(base + sc.off_y); z = load_f32_bytes(base + sc.off_z);
  } else if ((sc.stride_bytes & 15) == 0 && (reinterpret_cast<uintptr_t>(sc.pts) & 15) == 0) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(base));
    x = v.x; y = v.y; z = v.z;
  } else {
    const float* f = reinterpret_cast<const float*>(base);
    x = __ldg(f); y = __ldg(f + 1); z = __ldg(f + 2);
  }
}
__device__ __forceinline__ float4 load_xyzi(const ScanDesc& sc, int i) {
  const char* base = point_base(sc, i);
  float4 v;
  if (sc.generic) {
    v.x = load_f32_bytes(base + sc.off_x); v.y = load_f32_bytes(base + sc.off_y); v.z = load_f32_bytes(base + sc.off_z);
    v.w = sc.off_i >= 0 ? load_f32_bytes(base + sc.off_i) : 0.f;
    return v;
  }
  // pcl::PointXYZI keeps intensity in the second 16-byte half (data_c[0]); packed records at +12.
  const int ioff = sc.stride_bytes >= 32 ? 16 : 12;
  if ((sc.stride_bytes & 15) == 0 && (reinterpret_cast<uintptr_t>(sc.pts) & 15) == 0) {
    v = __ldg(reinterpret_cast<const float4*>(base));
    if (ioff != 12) v.w = __ldg(reinterpret_cast<const float*>(base + ioff));
  } else {
    const float* f = reinterpret_cast<const float*>(base);
    v.x = __ldg(f); v.y = __ldg(f + 1); v.z = __ldg(f + 2);
    v.w = sc.stride_bytes >= 16 ? __ldg(reinterpret_cast<const float*>(base + ioff)) : 0.f;
  }
  return v;
}

// Device atan is <= 2 ulp, glibc <= 1 ulp; after *180/pi and the affine bin map the two can differ by
// < 1e-13 in `v`. Decisions closer than kAmbTol to a boundary are counted as ambiguous.
constexpr double kAmbTol = 1e-12;
__device__ __forceinline__ bool near_int(double v) { return fabs(v - rint(v)) < kAmbTol; }

// Returns ring id or -1. `amb` is set when a bin decision sits within kAmbTol of a boundary
// (such a point could land in the other bin under a different libm).
// FP32 screening of the same decisions: when every comparison of the reference's double arithmetic (range
// gates, branch and reject thresholds, bin truncation) is further from its threshold than the FP32 error can
// reach, the float result IS the double result and the ~100 FP64 operations (sqrt, division, atan) are skipped.
// Error budget: sqrtf / division / atanf are within 2 ulp each, so the angle is within 1e-6 rad = 6e-5 deg and the
// bin coordinate v (slope <= 3 per degree) within 2e-4; the margins below are 5x that.  Returns false when a
// decision is too close to call (then the double path decides, as before).
__device__ __forceinline__ bool ring_of_point_fast(const DevParams& p, const ScanDesc& sc, int i, float xf, float yf, float zf, int* id_out) {
  const float d = sqrtf(xf * xf + yf * yf);
  const float minr = (float)p.min_range, maxr = (float)p.max_range;
  if (!(isfinite(xf) && isfinite(yf) && isfinite(zf))) { *id_out = -1; return true; }
  const float mr = 1e-3f;                                   // metres; float error at 75 m is 1e-5
  if (fabsf(d - minr) < mr || fabsf(d - maxr) < mr) return false;
  if (d > maxr || d < minr) { *id_out = -1; return true; }
  if (p.lidar_type == 1) { const int row = i / sc.width; *id_out = row < p.scan_lines ? row : -1; return true; }
  const float ang = atanf(zf / d) * 57.295779513f;
  const float ma = 3e-4f, mv = 1e-3f;
  int id;
  if (p.scan_lines == 64) {
    if (fabsf(ang + 8.83f) < ma || fabsf(ang - 2.0f) < ma || fabsf(ang + 24.33f) < ma) return false;
    if (ang > 2.0f || ang < -24.33f) { *id_out = -1; return true; }
    const float v = ang >= -8.83f ? (2.0f - ang) * 3.0f + 0.5f : (-8.83f - ang) * 2.0f + 0.5f;
    if (fabsf(v - rintf(v)) < mv) return false;
    id = (ang >= -8.83f ? 0 : 32) + (int)v;
    if (id > 63 || id < 0) id = -1;
  } else if (p.scan_lines == 32) {
    const float v = (ang + 30.666666f) * 0.75f;
    if (fabsf(v - rintf(v)) < mv) return false;
    id = (int)v;
    if (id > 31 || id < 0) id = -1;
  } else if (p.scan_lines == 16) {
    const float v = (ang + 15.0f) * 0.5f + 0.5f;
    if (fabsf(v - rintf(v)) < mv) return false;
    id = (int)v;
    if (id > 15 || id < 0) id = -1;
  } else {
    return false;
  }
  *id_out = id;
  return true;
}

// The reference's double arithmetic, for the points the FP32 screen cannot call.  Not inlined: the split kernels
// unroll their point loop eight times, and eight copies of the FP64 sqrt / division / atan made k_split_count 5000
// instructions long (instruction-cache misses: 3 warps per issue stalled on `no_instruction`).
// (scalars by value: a reference to the parameter structs would force a local-memory copy of them in the caller)
__device__ __noinline__ int ring_of_point_exact(double min_range, double max_range, int lidar_type, int scan_lines, int width, int i,
                                                float xf, float yf, float zf, bool* amb_out) {
  bool amb;
  const double x = xf, y = yf, z = zf;
  bool valid = isfinite(x) && isfinite(y) && isfinite(z);
  const double dist = sqrt(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)));
  if (dist > max_range || dist < min_range) valid = false;
  amb = false;
  *amb_out = false;
  if (!valid) return -1;
  if (lidar_type == 1) {
    const int row = i / width;
    return row < scan_lines ? row : -1;
  }
  const double angle = __ddiv_rn(__dmul_rn(atan(__ddiv_rn(z, dist)), 180.0), 3.14159265358979323846);
  int id = -1;
  if (scan_lines == 64) {
    double v;
    if (angle >= -8.83) { v = __dadd_rn(__dmul_rn(__dsub_rn(2.0, angle), 3.0), 0.5); id = __double2int_rz(v); }
    else { v = __dadd_rn(__dmul_rn(__dsub_rn(-8.83, angle), 2.0), 0.5); id = 32 + __double2int_rz(v); }
    amb = near_int(v) || fabs(angle - 2.0) < kAmbTol || fabs(angle + 24.33) < kAmbTol;
    if (fabs(angle + 8.83) < kAmbTol) {  // branch boundary: ambiguous only if the two formulas disagree
      const int hi = __double2int_rz(__dadd_rn(__dmul_rn(__dsub_rn(2.0, angle), 3.0), 0.5));
      const int lo = 32 + __double2int_rz(__dadd_rn(__dmul_rn(__dsub_rn(-8.83, angle), 2.0), 0.5));
      amb = amb || hi != lo;
    }
    if (angle > 2.0 || angle < -24.33 || id > 63 || id < 0) id = -1;
  } else if (scan_lines == 32) {
    const double v = __ddiv_rn(__dmul_rn(__dadd_rn(angle, 92.0 / 3.0), 3.0), 4.0);
    id = __double2int_rz(v); amb = near_int(v);
    if (id > 31 || id < 0) id = -1;
  } else if (scan_lines == 16) {
    const double v = __dadd_rn(__ddiv_rn(__dadd_rn(angle, 15.0), 2.0), 0.5);
    id = __double2int_rz(v); amb = near_int(v);
    if (id > 15 || id < 0) id = -1;
  }
  *amb_out = amb;
  return id;
}

__device__ __forceinline__ int ring_of_point(const DevParams& p, const ScanDesc& sc, int i, float xf, float yf, float zf, bool& amb) {
  int fast_id;
  if (ring_of_point_fast(p, sc, i, xf, yf, zf, &fast_id)) { amb = false; return fast_id; }
  return ring_of_point_exact(p.min_range, p.max_range, p.lidar_type, p.scan_lines, sc.width, i, xf, yf, zf, &amb);
}

// Pass 1: ring id per point + per-chunk histogram. grid (chunks, B), 256 threads, each warp
// owns a contiguous 256-point segment so that (warp, round, lane) is input order.
__global__ void __launch_bounds__(256) k_split_count(DevBuffers d, int lane0) {
  const int lane_b = lane_at(d, lane0 + blockIdx.y), chunk = blockIdx.x;
  const ScanDesc sc = d.scan[lane_b];
  const DevParams& p = d.p;
  const int L = p.scan_lines;
  __shared__ int hist[kMaxLines];
  __shared__ int s_amb;
  if (threadIdx.x < kMaxLines) hist[threadIdx.x] = 0;
  if (threadIdx.x == 0) s_amb = 0;
  __syncthreads();
  const int base = chunk * kChunk;
  if (base < sc.n) {
    const int w = threadIdx.x >> 5, ln = threadIdx.x & 31;
    uint8_t* rid = d.ring_id + (size_t)lane_b * p.Ncap;
    int namb = 0;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const int i = base + w * 256 + r * 32 + ln;
      int id = -1;
      if (i < sc.n) {
        float x, y, z; load_xyz(sc, i, x, y, z);
        bool amb; id = ring_of_point(p, sc, i, x, y, z, amb);
        namb += amb ? 1 : 0;
        rid[i] = id < 0 ? (uint8_t)255 : (uint8_t)id;
      }
      const unsigned m = __match_any_sync(0xffffffffu, id);
      if (id >= 0 && (__ffs(m) - 1) == ln) atomicAdd(&hist[id], __popc(m));
    }
    if (namb) atomicAdd(&s_amb, namb);
  }
  __syncthreads();
  int* out = d.chunk_hist + ((size_t)lane_b * p.chunks + chunk) * L;
  if (threadIdx.x < L) out[threadIdx.x] = hist[threadIdx.x];
  if (threadIdx.x == 0) d.chunk_amb[(size_t)lane_b * p.chunks + chunk] = s_amb;
}

// Pass 2: exclusive scan over (ring-major, chunk) -> chunk_base, ring_off. grid B, 128 threads.
// One thread per ring walks that ring's chunk counts; the loads are issued eight at a time (their addresses do not
// depend on the running sum), which turns ~60 dependent round trips into ~8 (21 -> 5 us at 128 lanes).
__global__ void __launch_bounds__(kMaxLines) k_split_scan(DevBuffers d, int lane0) {
  const int lane_b = lane_at(d, lane0 + blockIdx.x);
  const DevParams& p = d.p;
  const int L = p.scan_lines, r = threadIdx.x;
  const ScanDesc sc = d.scan[lane_b];
  const int nch = (sc.n + kChunk - 1) / kChunk;
  __shared__ int tot[kMaxLines + 1];
  __shared__ int s_amb;
  if (r == 0) s_amb = 0;
  __syncthreads();
  int run = 0;
  if (r < L) {
    const int* h = d.chunk_hist + (size_t)lane_b * p.chunks * L + r;
    int* b = d.chunk_base + (size_t)lane_b * p.chunks * L + r;
    for (int c0 = 0; c0 < nch; c0 += 8) {
      int v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = c0 + k < nch ? h[(size_t)(c0 + k) * L] : 0;
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (c0 + k < nch) { b[(size_t)(c0 + k) * L] = run; run += v[k]; }
    }
    tot[r] = run;
  }
  {   // ambiguous-bin count of the scan: every thread sums a strided share of the chunks
    int amb = 0;
    for (int c = r; c < nch; c += blockDim.x) amb += d.chunk_amb[(size_t)lane_b * p.chunks + c];
    if (amb) atomicAdd(&s_amb, amb);
  }
  __syncthreads();
  if (r == 0) {
    int acc = 0;
    int* off = d.ring_off + (size_t)lane_b * (L + 1);
    for (int k = 0; k < L; ++k) { off[k] = acc; acc += tot[k]; }
    off[L] = acc;
    d.ostate[lane_b].n_valid = acc;
    d.ostate[lane_b].n_ambiguous = s_amb;
  }
}

// Pass 3: stable scatter into ring-major order. grid (chunks, B), 256 threads.
__global__ void __launch_bounds__(256) k_split_scatter(DevBuffers d, int lane0) {
  // CTAs walk the lane list in the REVERSE of k_split_count's order: the scans that pass read last are still in L2
  const int lane_b = lane_at(d, lane0 + (int)(gridDim.y - 1u - blockIdx.y)), chunk = (int)(gridDim.x - 1u - blockIdx.x);
  const ScanDesc sc = d.scan[lane_b];
  const DevParams& p = d.p;
  const int L = p.scan_lines;
  const int base = chunk * kChunk;
  if (base >= sc.n) return;
  __shared__ int wcnt[8][kMaxLines];
  for (int k = threadIdx.x; k < 8 * kMaxLines; k += 256) (&wcnt[0][0])[k] = 0;
  __syncthreads();
  const int w = threadIdx.x >> 5, ln = threadIdx.x & 31;
  const uint8_t* rid = d.ring_id + (size_t)lane_b * p.Ncap;
  int ids[8];
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int i = base + w * 256 + r * 32 + ln;
    int id = -1;
    if (i < sc.n) { const uint8_t v = rid[i]; id = v == 255 ? -1 : (int)v; }
    ids[r] = id;
    const unsigned m = __match_any_sync(0xffffffffu, id);
    if (id >= 0 && (__ffs(m) - 1) == ln) wcnt[w][id] += __popc(m);
    __syncwarp();
  }
  __syncthreads();
  if (threadIdx.x < L) {
    const int r = threadIdx.x;
    int run = d.chunk_base[((size_t)lane_b * p.chunks + chunk) * L + r] + d.ring_off[(size_t)lane_b * (L + 1) + r];
#pragma unroll
    for (int ww = 0; ww < 8; ++ww) { const int c = wcnt[ww][r]; wcnt[ww][r] = run; run += c; }
  }
  __syncthreads();
  float4* rings = d.rings + (size_t)lane_b * p.Ncap;
  int* src = d.src_index ? d.src_index + (size_t)lane_b * p.Ncap : nullptr;
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int i = base + w * 256 + r * 32 + ln;
    const int id = ids[r];
    const unsigned m = __match_any_sync(0xffffffffu, id);
    if (id >= 0) {
      const int pos = wcnt[w][id] + __popc(m & ((1u << ln) - 1u));
      rings[pos] = load_xyzi(sc, i);
      if (src) src[pos] = i;
    }
    __syncwarp();
    if (id >= 0 && (__ffs(m) - 1) == ln) wcnt[w][id] += __popc(m);
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------
// A3 + A4: curvature and greedy selection, one CTA per (ring, lane).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

// 11-tap sum in float, strictly left to right, 10*x a separate float multiply
// (src/feature_extractor.cc:196-228).
__device__ __forceinline__ float tap11(float m5, float m4, float m3, float m2, float m1, float c,
                                       float p1, float p2, float p3, float p4, float p5) {
  float s = __fadd_rn(m5, m4);
  s = __fadd_rn(s, m3); s = __fadd_rn(s, m2); s = __fadd_rn(s, m1);
  s = __fsub_rn(s, __fmul_rn(10.0f, c));
  s = __fadd_rn(s, p1); s = __fadd_rn(s, p2); s = __fadd_rn(s, p3); s = __fadd_rn(s, p4); s = __fadd_rn(s, p5);
  return s;
}

// squared gap between consecutive ring points a, b (src/feature_extractor.cc:281-289):
// float differences widened to double, then dx*dx + dy*dy + dz*dz in double.
__device__ __forceinline__ double gap2(const float4& a, const float4& b) {
  const double dx = (double)__fsub_rn(a.x, b.x), dy = (double)__fsub_rn(a.y, b.y), dz = (double)__fsub_rn(a.z, b.z);
  return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

struct RingView {
  const float4* P;    // ring points (shared or global)
  const double* K;    // smoothness per ring index
  unsigned* bits;     // picked bitmap over ring indices
  int n;
};

__device__ __forceinline__ bool bit_get(const unsigned* bits, int i) { return (((const volatile unsigned*)bits)[i >> 5] >> (i & 31)) & 1u; }
__device__ __forceinline__ void bit_set(unsigned* bits, int i) { atomicOr(&bits[i >> 5], 1u << (i & 31)); }

// Mark idx and its +-5 neighbourhood (gap-limited) into `bits`, restricted to [lo, hi).
// Executed by one full warp: lanes 0-4 test the forward gaps, lanes 8-12 the backward gaps.
__device__ __forceinline__ void mark_pick(const RingView& rv, unsigned* bits, int idx, int lo, int hi, int ln) {
  bool brk = false;
  if (ln < 5) { const int l = ln + 1; brk = gap2(rv.P[idx + l], rv.P[idx + l - 1]) > 0.05; }
  else if (ln >= 8 && ln < 13) { const int l = ln - 7; brk = gap2(rv.P[idx - l], rv.P[idx - l + 1]) > 0.05; }
  const unsigned bm = __ballot_sync(0xffffffffu, brk);
  const unsigned f = bm & 0x1fu, b = (bm >> 8) & 0x1fu;
  const int nf = f ? (__ffs(f) - 1) : 5, nb = b ? (__ffs(b) - 1) : 5;  // marks before the first break
  if (ln == 0) { if (idx >= lo && idx < hi) bit_set(bits, idx); }
  if (ln >= 1 && ln <= nf) { const int j = idx + ln; if (j >= lo && j < hi) bit_set(bits, j); }
  if (ln >= 9 && ln <= 8 + nb) { const int j = idx - (ln - 8); if (j >= lo && j < hi) bit_set(bits, j); }
  __syncwarp();
}

// Forward suppression of a region's picks beyond its end `hi` (src/feature_extractor.cc:280-294):
// bit b set <=> ring index hi + b is marked by a pick of this region.  Warp-uniform result.
__device__ __forceinline__ unsigned region_spill(const RingView& rv, const int* picks, int np, int hi, int ln) {
  unsigned m = 0;
  for (int k = ln; k < np; k += 32) {
    const int idx = picks[k];
    if (idx + 5 >= hi && hi + 4 < rv.n) {
      for (int l = 1; l <= 5; ++l) {
        if (gap2(rv.P[idx + l], rv.P[idx + l - 1]) > 0.05) break;
        if (idx + l >= hi) m |= 1u << (idx + l - hi);
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m |= __shfl_xor_sync(0xffffffffu, m, o);
  return m;
}

// Greedy selection of one region by one warp: repeated warp-shuffle arg-max over the
// not-yet-picked items under the total order (smoothness desc, index asc). Equivalent to
// std::sort + walk of src/feature_extractor.cc:261-312 whenever the sort order is total.
__device__ int run_region(const RingView& rv, int lo, int hi, int epr, int* picks, int ln) {
  int np = 0;
  for (;;) {
    double bk = -1.0; int bi = 0x7fffffff;
    for (int i = lo + ln; i < hi; i += 32)
      if (!bit_get(rv.bits, i)) { const double k = rv.K[i]; if (k > bk) { bk = k; bi = i; } }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ok = __shfl_xor_sync(0xffffffffu, bk, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ok > bk || (ok == bk && oi < bi)) { bk = ok; bi = oi; }
    }
    if (bi == 0x7fffffff) break;            // every item already picked
    if (bk < 0.1 || np > epr) break;        // src/feature_extractor.cc:270
    if (ln == 0) picks[np] = bi;
    ++np;
    mark_pick(rv, rv.bits, bi, lo, hi, ln);
  }
  return np;
}

// Five consecutive bits of the gap bitmap starting at ring index p (bit k = "points p+k and p+k+1 are more than
// sqrt(0.05) m apart", src/feature_extractor.cc:281-291): bit 0 is index p.
__device__ __forceinline__ unsigned gap5(const unsigned* gapbits, int p, int wcap) {
  const int w0 = p >> 5;
  const unsigned a = gapbits[w0], b = w0 + 1 < wcap ? gapbits[w0 + 1] : 0u;
  return __funnelshift_r(a, b, p & 31) & 0x1fu;
}

// Forward suppression of a region's picks beyond its end `hi`, from the gap bitmap (see region_spill).
__device__ __forceinline__ unsigned region_spill_fast(const unsigned* gapbits, int wcap, const int* picks, int np, int hi, int n, int ln) {
  unsigned m = 0;
  for (int k = ln; k < np; k += 32) {
    const int idx = picks[k];
    if (idx + 5 >= hi && hi + 4 < n) {
      const unsigned f = gap5(gapbits, idx, wcap);
      const int nf = f ? (__ffs(f) - 1) : 5;
      for (int l = 1; l <= nf; ++l)
        if (idx + l >= hi) m |= 1u << (idx + l - hi);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m |= __shfl_xor_sync(0xffffffffu, m, o);
  return m;
}

// Register-cached variant for regions of at most 256 items (8 per lane): keys and availability live in registers.
// The +-5 suppression reads the precomputed gap bitmap (one bit per consecutive pair of ring points, filled once per
// ring with every lane busy) instead of evaluating ten FP64 gaps per pick in ten lanes; the warp arg-max is three
// redux operations on the order-preserving integer image of the non-negative key (high word, low word among ties,
// lowest index among ties) instead of five 96-bit shuffle rounds.
// `premask`: bit b set <=> ring index lo + b is already suppressed by the previous region's picks.
// Same selection as run_region (total order smoothness desc, index asc).
__device__ int run_region_reg(const RingView& rv, const unsigned* gapbits, int wcap, int lo, int hi, int epr, int* picks, int ln, unsigned premask) {
  double kk[8];
  unsigned dead = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int i = lo + ln + 32 * j;
    kk[j] = i < hi ? rv.K[i] : -1.0;
    if (i >= hi || (i - lo < 5 && ((premask >> (i - lo)) & 1u))) dead |= 1u << j;
  }
  int np = 0;
  for (;;) {
    double bk = -1.0; int bi = 0x7fffffff;
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (!((dead >> j) & 1u) && kk[j] > bk) { bk = kk[j]; bi = lo + ln + 32 * j; }
    // keys are sums of squares (>= +0): their bit patterns order like the values; a lane without a live item offers 0
    const unsigned long long kb = bi == 0x7fffffff ? 0ull : (unsigned long long)__double_as_longlong(bk);
    const unsigned khi = (unsigned)(kb >> 32), klo = (unsigned)kb;
    const unsigned mh = __reduce_max_sync(0xffffffffu, khi);
    const unsigned ml = __reduce_max_sync(0xffffffffu, khi == mh ? klo : 0u);
    bi = (int)__reduce_min_sync(0xffffffffu, (khi == mh && klo == ml) ? (unsigned)bi : 0x7fffffffu);
    bk = __longlong_as_double((long long)(((unsigned long long)mh << 32) | ml));
    if (bi == 0x7fffffff) break;            // every item already picked
    if (bk < 0.1 || np > epr) break;        // src/feature_extractor.cc:270
    if (ln == 0) picks[np] = bi;
    ++np;
    // +-5 suppression, gap-limited (src/feature_extractor.cc:280-310)
    const unsigned f = gap5(gapbits, bi, wcap), bb = gap5(gapbits, bi - 5, wcap);
    const int nf = f ? (__ffs(f) - 1) : 5;                // forward: stop before the first wide gap
    const int nb = bb ? (__clz(bb) - 27) : 5;             // backward: bit 4 is the pair (bi-1, bi); highest set bit h -> 4 - h
    const int first = bi - nb;
    const int i = first + ((ln - (first - lo)) & 31);     // this lane's only index in [first, first + 32)
    if (i <= bi + nf && i >= lo && i < hi) dead |= 1u << ((i - lo) >> 5);
  }
  return np;
}

// NT: threads per CTA.  256 for rings that fit shared memory (4 CTAs per SM); 1024 when the expected ring is longer
// than the shared-memory capacity (1M-point scans: 15,625 points per ring, one CTA per ring is all the parallelism
// there is, so the CTA should be as wide as possible: 32 warps for the curvature and the 64 regions).
template <int NT>
__global__ void __launch_bounds__(NT, NT == 256 ? 4 : 1) k_extract(DevBuffers d, int lane0, int ring_cap, int want_keys, int ring0) {
  const DevParams& p = d.p;
  const int lane_b = lane_at(d, lane0 + blockIdx.y), ring = ring0 + blockIdx.x;   // ring0 > 0: ring-sharded extraction
  const int L = p.scan_lines, R = p.scan_regions, epr = p.edges_per_region, E1 = epr + 1;
  const int* roff = d.ring_off + (size_t)lane_b * (L + 1);
  const int off = roff[ring], n = roff[ring + 1] - off;
  int* rcnt = d.region_cnt + ((size_t)lane_b * L + ring) * R;
  const int tid = threadIdx.x, ln = tid & 31, w = tid >> 5;
  if (n < R * epr + 10) {  // min_points_per_scan_ (src/params.cc:63, src/feature_extractor.cc:188)
    for (int r = tid; r < R; r += blockDim.x) rcnt[r] = 0;
    return;
  }
  extern __shared__ __align__(128) unsigned char smem[];
  // layout: [points ring_cap*16][keys ring_cap*8][bits][tbits][picks R*E1][npicks R]
  float4* sp = reinterpret_cast<float4*>(smem);
  double* sk = reinterpret_cast<double*>(smem + (size_t)ring_cap * 16);
  const bool in_smem = n <= ring_cap;
  const int nwords = (n + 31) >> 5;
  const int wcap = (ring_cap + 31) >> 5;
  unsigned* sbits = reinterpret_cast<unsigned*>(smem + (size_t)ring_cap * 24);
  unsigned* stbits = sbits + wcap;
  int* picks = reinterpret_cast<int*>(stbits + wcap);
  int* npicks = picks + R * E1;
  __shared__ __align__(8) unsigned long long mbar;

  const float4* gp = d.rings + (size_t)lane_b * p.Ncap + off;
  RingView rv;
  rv.n = n;
  if (in_smem) {
    // TMA bulk copy of the whole ring (n*16 bytes, 16-byte aligned) into shared memory.
    const unsigned bytes = (unsigned)n * 16u;
    if (tid == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mbar)));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&mbar)), "r"(bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"(smem_u32(sp)), "l"(gp), "r"(bytes), "r"(smem_u32(&mbar)) : "memory");
    }
    for (int k = tid; k < wcap; k += blockDim.x) sbits[k] = 0u;  // overlap with the copy (the gap bitmap behind it is written whole)
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(smem_u32(&mbar)), "r"(0) : "memory");
    rv.P = sp; rv.K = sk; rv.bits = sbits;
  } else {
    // Long ring (e.g. the 1M-point scan): points stay in global/L2, keys and bitmaps in
    // global scratch. Bitmap words [off/32 + ring, ...) are disjoint between rings.
    double* gk = d.keys + (size_t)lane_b * p.Ncap + off;
    const size_t bw = (size_t)(p.Ncap >> 5) + kMaxLines + 2;
    unsigned* gbits = d.pick_bits + (size_t)lane_b * 2 * bw + (off >> 5) + ring;
    unsigned* gtbits = gbits + bw;
    for (int k = tid; k < nwords; k += blockDim.x) { gbits[k] = 0u; gtbits[k] = 0u; }
    rv.P = gp; rv.K = gk; rv.bits = gbits;
    stbits = gtbits;
    sk = gk;
  }
  // curvature
  double* gkeys = (want_keys && d.keys) ? d.keys + (size_t)lane_b * p.Ncap + off : nullptr;
  if (in_smem) {
    // Every thread takes runs of kRun CONSECUTIVE points and slides an 11-point window through registers: 10 + kRun
    // shared-memory loads per run instead of 11 per point.  kRun = 9: the lanes' float4 reads are 144 bytes apart,
    // which keeps a quarter-warp on distinct banks (a power-of-two run length would put all eight on the same four).
    constexpr int kRun = 9;
    for (int r0 = tid * kRun; r0 < n - 10; r0 += blockDim.x * kRun) {
      const int j0 = 5 + r0;
      float wx[11], wy[11], wz[11];
#pragma unroll
      for (int k = 0; k < 10; ++k) { const float4 v = sp[j0 - 5 + k]; wx[k] = v.x; wy[k] = v.y; wz[k] = v.z; }
#pragma unroll
      for (int q = 0; q < kRun; ++q) {
        const int j = j0 + q;
        const float4 v = sp[min(j + 5, n - 1)];
        wx[10] = v.x; wy[10] = v.y; wz[10] = v.z;
        const double dx = (double)tap11(wx[0], wx[1], wx[2], wx[3], wx[4], wx[5], wx[6], wx[7], wx[8], wx[9], wx[10]);
        const double dy = (double)tap11(wy[0], wy[1], wy[2], wy[3], wy[4], wy[5], wy[6], wy[7], wy[8], wy[9], wy[10]);
        const double dz = (double)tap11(wz[0], wz[1], wz[2], wz[3], wz[4], wz[5], wz[6], wz[7], wz[8], wz[9], wz[10]);
        const double key = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
        if (j < n - 5) {
          sk[j] = key;
          if (gkeys) gkeys[j] = key;
        }
#pragma unroll
        for (int k = 0; k < 10; ++k) { wx[k] = wx[k + 1]; wy[k] = wy[k + 1]; wz[k] = wz[k + 1]; }
      }
    }
  } else
  for (int j = 5 + tid; j < n - 5; j += blockDim.x) {
    const float4 a0 = rv.P[j - 5], a1 = rv.P[j - 4], a2 = rv.P[j - 3], a3 = rv.P[j - 2], a4 = rv.P[j - 1];
    const float4 c = rv.P[j];
    const float4 b1 = rv.P[j + 1], b2 = rv.P[j + 2], b3 = rv.P[j + 3], b4 = rv.P[j + 4], b5 = rv.P[j + 5];
    const double dx = (double)tap11(a0.x, a1.x, a2.x, a3.x, a4.x, c.x, b1.x, b2.x, b3.x, b4.x, b5.x);
    const double dy = (double)tap11(a0.y, a1.y, a2.y, a3.y, a4.y, c.y, b1.y, b2.y, b3.y, b4.y, b5.y);
    const double dz = (double)tap11(a0.z, a1.z, a2.z, a3.z, a4.z, c.z, b1.z, b2.z, b3.z, b4.z, b5.z);
    const double key = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
    sk[j] = key;
    if (gkeys && in_smem) gkeys[j] = key;
  }
  if (in_smem) {
    // gap bitmap: bit j <=> consecutive ring points j, j+1 are more than sqrt(0.05) m apart (the +-5 suppression's
    // break test, src/feature_extractor.cc:281-291 / :297-307: the same squared gap in both directions)
    for (int base = tid & ~31; base < n; base += blockDim.x) {
      const int j = base + ln;
      const bool g = j + 1 < n && gap2(rv.P[j + 1], rv.P[j]) > 0.05;
      const unsigned word = __ballot_sync(0xffffffffu, g);
      if (ln == 0) stbits[base >> 5] = word;
    }
  }
  __syncthreads();

  const int total = n - 10, sector = total / R;
  const int nw = blockDim.x >> 5;
  // regions of <= 256 items of a ring held in shared memory take the register-cached path
  const bool fast = in_smem && (sector + R) <= 256;
  __shared__ unsigned s_spill[256];   // per region: suppression spilled into the next region (5 bits)
  // speculative pass: every region on its own (no premask), marks confined to the region
  for (int r = w; r < R; r += nw) {
    const int lo = sector * r + 5, hi = (r == R - 1 ? total : sector * (r + 1)) + 5;
    const int np = fast ? run_region_reg(rv, stbits, wcap, lo, hi, epr, picks + r * E1, ln, 0u) : run_region(rv, lo, hi, epr, picks + r * E1, ln);
    if (ln == 0) npicks[r] = np;
    __syncwarp();
    const unsigned sp = fast ? region_spill_fast(stbits, wcap, picks + r * E1, np, hi, n, ln) : region_spill(rv, picks + r * E1, np, hi, ln);
    if (ln == 0) s_spill[r] = sp;
  }
  __syncthreads();
  // The only coupling between the regions of a ring is picked_: a pick within 5 points of the end of
  // region r suppresses (gap-limited) up to 5 points beyond it.  Each region's spill is a 5-bit mask
  // over the indices that follow it; `carry` accumulates the spills of the regions behind, shifted to the
  // current region's start (regions shorter than 5 points — edges_per_region < 5 — pass part of a spill on
  // to their successors).  A region is re-run only if one of its speculative picks is suppressed by the
  // (final) carry.  Warp 0 walks the regions in order; without clashes this is O(R) checks.
  if (w == 0) {
    unsigned carry = 0;        // bit b: ring index lo_r + b is suppressed by a pick of an earlier region
    for (int r = 0; r < R; ++r) {
      const int lo = sector * r + 5, hi = (r == R - 1 ? total : sector * (r + 1)) + 5;
      const unsigned spill_prev = carry & 0x1fu;
      int np = npicks[r];
      bool rerun = false;
      if (spill_prev) {
        bool clash = false;
        for (int k = ln; k < np; k += 32) { const int o = picks[r * E1 + k] - lo; clash |= o < 5 && ((spill_prev >> o) & 1u); }
        rerun = __any_sync(0xffffffffu, clash);
      }
      if (rerun) {
        if (fast) np = run_region_reg(rv, stbits, wcap, lo, hi, epr, picks + r * E1, ln, spill_prev);
        else {
          // rerun with the true premask: clear the region's bits, set the spilled ones
          for (int i = (lo >> 5) + ln; i <= ((hi - 1) >> 5); i += 32) {
            unsigned m = 0xffffffffu;
            if (i == (lo >> 5)) m &= 0xffffffffu << (lo & 31);
            if (i == ((hi - 1) >> 5)) m &= 0xffffffffu >> (31 - ((hi - 1) & 31));
            atomicAnd(&rv.bits[i], ~m);
          }
          __syncwarp();
          if (ln < 5 && ((spill_prev >> ln) & 1u) && lo + ln < hi) bit_set(rv.bits, lo + ln);
          __syncwarp();
          np = run_region(rv, lo, hi, epr, picks + r * E1, ln);
        }
        if (ln == 0) npicks[r] = np;
        __syncwarp();
      }
      const unsigned spill_out = !rerun ? s_spill[r] : (fast ? region_spill_fast(stbits, wcap, picks + r * E1, np, hi, n, ln) : region_spill(rv, picks + r * E1, np, hi, ln));
      carry = ((hi - lo) >= 32 ? 0u : (carry >> (hi - lo))) | spill_out;
    }
  }
  __syncthreads();
  // emit into fixed (ring, region, pick) slots
  float4* slots = d.slots + (size_t)lane_b * p.Ecap + (size_t)ring * R * E1;
  int* sidx = d.slot_idx + (size_t)lane_b * p.Ecap + (size_t)ring * R * E1;
  for (int s = tid; s < R * E1; s += blockDim.x) {
    const int r = s / E1, k = s - r * E1;
    if (k < npicks[r]) { const int j = picks[s]; slots[s] = rv.P[j]; sidx[s] = j; }
  }
  for (int r = tid; r < R; r += blockDim.x) rcnt[r] = npicks[r];
}

// Compaction of the fixed slots into the contiguous edge list (ring, region, pick order).  Two CTAs per SM (32
// registers): left free, ptxas spends 42 registers on it once the lane comes from the lane list.
__global__ void __launch_bounds__(1024, 2) k_compact(DevBuffers d, int lane0) {
  const DevParams& p = d.p;
  const int lane_b = lane_at(d, lane0 + blockIdx.x), tid = threadIdx.x;
  const int LR = p.scan_lines * p.scan_regions, E1 = p.edges_per_region + 1;
  extern __shared__ int base[];  // LR + 32
  int* wsum = base + LR;
  const int* rcnt = d.region_cnt + (size_t)lane_b * LR;
  const int per = (LR + 1023) / 1024;
  int local = 0;
  for (int k = 0; k < per; ++k) { const int i = tid * per + k; if (i < LR) local += rcnt[i]; }
  int inc = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, inc, o); if ((tid & 31) >= o) inc += v; }
  if ((tid & 31) == 31) wsum[tid >> 5] = inc;
  __syncthreads();
  if (tid < 32) {
    int v = wsum[tid], s = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, s, o); if (tid >= o) s += u; }
    wsum[tid] = s - v;
    if (tid == 31) { d.ostate[lane_b].n_edges = s; d.diag[lane_b].n_edges = s; }
  }
  __syncthreads();
  int run = wsum[tid >> 5] + inc - local;
  for (int k = 0; k < per; ++k) { const int i = tid * per + k; if (i < LR) { base[i] = run; run += rcnt[i]; } }
  __syncthreads();
  const float4* slots = d.slots + (size_t)lane_b * p.Ecap;
  const int* sidx = d.slot_idx + (size_t)lane_b * p.Ecap;
  float4* edges = d.edges + (size_t)lane_b * p.Ecap;
  int* ering = d.edge_ring + (size_t)lane_b * p.Ecap;
  int* eidx = d.edge_idx + (size_t)lane_b * p.Ecap;
  for (int s = tid; s < LR * E1; s += 1024) {
    const int rr = s / E1, k = s - rr * E1;
    if (k < rcnt[rr]) {
      const int o = base[rr] + k;
      edges[o] = slots[s]; ering[o] = rr / p.scan_regions; eidx[o] = sidx[s];
    }
  }
}

static size_t extract_smem_bytes(const DevParams& p, int ring_cap) {
  const int wcap = (ring_cap + 31) >> 5;
  return (size_t)ring_cap * 24 + (size_t)wcap * 8 + (size_t)p.scan_regions * (p.edges_per_region + 1) * 4 + (size_t)p.scan_regions * 4 + 16;
}

// Ring points kept in shared memory by k_extract.  The kernel alternates block-wide phases (curvature, per-warp
// region selection, a one-warp fix-up, emission), so resident CTAs per SM matter: the capacity is the largest one
// that still lets k CTAs share an SM's 228 KB, for the largest k whose capacity covers the expected ring length
// (max_points / scan_lines + 5 %; 4 CTAs/SM for HDL-64 and OS1-128: extract 0.44 -> 0.39 ms/step at 128 lanes).
// Longer rings are still handled, through the global-memory path.
int extract_ring_cap(const DevParams& p) {
  const long need = ((long)p.Ncap * 21 / 20) / p.scan_lines;
  const long fixed = (long)p.scan_regions * (p.edges_per_region + 1) * 4 + (long)p.scan_regions * 4 + 16 + 1024 /* s_spill */;
  long cap = kRingSmemCap;
  for (int k = 4; k >= 1; --k) {
    long ck = ((228L * 1024) / k - 2048 - fixed) * 4 / 97;   // 24 B per point + 2 bitmap bits per point = 24.25 B
    ck = ck / 32 * 32;
    if (ck > kRingSmemCap) ck = kRingSmemCap;
    if (ck >= need || k == 1) { cap = ck; break; }
  }
  if (cap < 1024) cap = 1024;
  return (int)cap;
}

// the expected ring (max_points / scan_lines + 5 %) does not fit the shared-memory ring buffer: global-memory path
static bool extract_long_rings(const DevParams& p, int ring_cap) { return ((long)p.Ncap * 21 / 20) / p.scan_lines > ring_cap; }

int launch_split(const DevBuffers& d, cudaStream_t s, LaneRange lr) {
  const dim3 g(d.p.chunks, lr.nlanes);
  k_split_count<<<g, 256, 0, s>>>(d, lr.lane0);
  k_split_scan<<<lr.nlanes, kMaxLines, 0, s>>>(d, lr.lane0);
  k_split_scatter<<<g, 256, 0, s>>>(d, lr.lane0);
  return 3;
}

// Dynamic shared memory above 48 KB is an opt-in PER DEVICE: liodom_ctx_create calls this after cudaSetDevice, so
// every device a context lives on gets the limit raised (to the architectural maximum: contexts with different
// parameters may share a device).  Returns the first CUDA error.
template <typename K>
static cudaError_t raise_dynamic_smem_limit(K kernel) {
  int dev = 0, optin = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  if (e != cudaSuccess) return e;
  cudaFuncAttributes fa;
  e = cudaFuncGetAttributes(&fa, kernel);
  if (e != cudaSuccess) return e;
  // the opt-in limit covers static + dynamic shared memory of a CTA
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)fa.sharedSizeBytes);
}
cudaError_t configure_extract_kernels() {
  cudaError_t e = raise_dynamic_smem_limit(k_extract<256>);
  if (e != cudaSuccess) return e;
  e = raise_dynamic_smem_limit(k_extract<1024>);
  if (e != cudaSuccess) return e;
  return raise_dynamic_smem_limit(k_compact);
}
size_t extract_smem_needed(const DevParams& p) {   // + 4 KB for the kernels' static shared memory
  const size_t a = extract_smem_bytes(p, extract_ring_cap(p)), b = (size_t)(p.scan_lines * p.scan_regions + 32) * sizeof(int);
  return (a > b ? a : b) + 4096;
}

int launch_extract_rings(const DevBuffers& d, cudaStream_t s, LaneRange lr, int ring0, int nrings) {
  const int ring_cap = extract_ring_cap(d.p);
  const size_t sm = extract_smem_bytes(d.p, ring_cap);
  if (extract_long_rings(d.p, ring_cap)) k_extract<1024><<<dim3(nrings, lr.nlanes), 1024, sm, s>>>(d, lr.lane0, ring_cap, 0, ring0);
  else k_extract<256><<<dim3(nrings, lr.nlanes), 256, sm, s>>>(d, lr.lane0, ring_cap, 0, ring0);
  return 1;
}
int launch_compact(const DevBuffers& d, cudaStream_t s, LaneRange lr) {
  const int LR = d.p.scan_lines * d.p.scan_regions;
  k_compact<<<lr.nlanes, 1024, (LR + 32) * sizeof(int), s>>>(d, lr.lane0);
  return 1;
}

int launch_extract(const DevBuffers& d, cudaStream_t s, LaneRange lr, bool want_keys) {
  const int ring_cap = extract_ring_cap(d.p);
  const size_t sm = extract_smem_bytes(d.p, ring_cap);
  if (extract_long_rings(d.p, ring_cap)) k_extract<1024><<<dim3(d.p.scan_lines, lr.nlanes), 1024, sm, s>>>(d, lr.lane0, ring_cap, want_keys ? 1 : 0, 0);
  else k_extract<256><<<dim3(d.p.scan_lines, lr.nlanes), 256, sm, s>>>(d, lr.lane0, ring_cap, want_keys ? 1 : 0, 0);
  const int LR = d.p.scan_lines * d.p.scan_regions;
  k_compact<<<lr.nlanes, 1024, (LR + 32) * sizeof(int), s>>>(d, lr.lane0);
  return 2;
}

}  // namespace liodom
