// On-device Levenberg-Marquardt on SE(3) for the weighted edge-to-line cost: replaces the
// Ceres problem of src/laser_odometry.cc:198-228 with the cost of
// include/liodom/factors.hpp:64-121 (Point2LineFactor), HuberLoss(0.2) and the
// EigenQuaternionParameterization tangent space.  One thread-block cluster per lane runs the
// whole solve: per-edge residual/Jacobian in FP64, fixed-order shuffle / shared / distributed-
// shared reduction to the 6x6 normal equations, trust-region controller (Ceres 1.14 defaults,
// SURVEY.md App. A.5) on thread 0 of the leading CTA.  Tolerance parity (1e-4 m / 1e-5 rad), so FMA contraction is allowed here.
#include "common.cuh"
#include <cooperative_groups.h>
#include <float.h>

namespace liodom {

constexpr int kSolveThreads = 256;
constexpr int kNumAcc = 29;  // 21 (upper H) + 6 (g) + cost + block count
constexpr int kValidCap = 8192;  // valid residual blocks a CTA can list in shared memory (beyond: the uncompacted loop)

struct LmCtrl {
  double x[7], xc[7];
  double H[21], g[6];
  double scale[6], diagonal[6];
  double radius, decrease_factor, x_cost, x_norm, gradient_max_norm, model_cost_change;
  int iteration, num_invalid, reuse_diagonal, step_is_successful, first;
  int action;  // 0: evaluate Jacobian at x, 1: evaluate cost at xc, 2: done
  SolveSummaryDev sum;
};

__device__ __forceinline__ int hidx(int i, int j) { return i * 6 - (i * (i - 1)) / 2 + (j - i); }  // i <= j

__device__ void quat_plus(const double* x, const double* dl, double* o) {
  const double n = sqrt(dl[0] * dl[0] + dl[1] * dl[1] + dl[2] * dl[2]);
  if (n > 0.0) {
    const double s = sin(n) / n;
    const double dw = cos(n), dx = s * dl[0], dy = s * dl[1], dz = s * dl[2];
    const double xw = x[3], xx = x[0], xy = x[1], xz = x[2];
    o[3] = dw * xw - dx * xx - dy * xy - dz * xz;
    o[0] = dw * xx + dx * xw + dy * xz - dz * xy;
    o[1] = dw * xy + dy * xw + dz * xx - dx * xz;
    o[2] = dw * xz + dz * xw + dx * xy - dy * xx;
  } else { o[0] = x[0]; o[1] = x[1]; o[2] = x[2]; o[3] = x[3]; }
}
__device__ void state_plus(const double* x, const double* d6, double* o) {
  quat_plus(x, d6, o);
  o[4] = x[4] + d6[3]; o[5] = x[5] + d6[4]; o[6] = x[6] + d6[5];
}

__device__ bool chol_solve6(const double* Hs, const double* D2, const double* gs, double* y) {
  double L[36];
  for (int i = 0; i < 6; ++i)
    for (int j = 0; j <= i; ++j) {
      double s = Hs[hidx(j, i)] + (i == j ? D2[i] : 0.0);
      for (int k = 0; k < j; ++k) s -= L[i * 6 + k] * L[j * 6 + k];
      if (i == j) { if (!(s > 0.0)) return false; L[i * 6 + i] = sqrt(s); }
      else L[i * 6 + j] = s / L[j * 6 + j];
    }
  double z[6];
  for (int i = 0; i < 6; ++i) { double s = gs[i]; for (int k = 0; k < i; ++k) s -= L[i * 6 + k] * z[k]; z[i] = s / L[i * 6 + i]; }
  for (int i = 5; i >= 0; --i) { double s = z[i]; for (int k = i + 1; k < 6; ++k) s -= L[k * 6 + i] * y[k]; y[i] = s / L[i * 6 + i]; }
  for (int k = 0; k < 6; ++k) if (!isfinite(y[k])) return false;
  return true;
}

__device__ void lm_done(LmCtrl& c, int termination) { c.sum.termination = termination; c.action = 2; }

// TrustRegionMinimizer loop body up to the next evaluation (thread 0 only).
__device__ void lm_try_step(LmCtrl& c) {
  for (;;) {
    if (c.iteration >= 4) return lm_done(c, 0);                                           // max_num_iterations
    if (c.step_is_successful && c.gradient_max_norm <= 1e-10) return lm_done(c, 1);        // gradient_tolerance
    if (c.radius < 1e-32) return lm_done(c, 5);                                            // min_trust_region_radius
    c.iteration++;
    double Hs[21], gs[6], D2[6];
    for (int i = 0; i < 6; ++i) { gs[i] = c.g[i] * c.scale[i]; for (int j = i; j < 6; ++j) Hs[hidx(i, j)] = c.H[hidx(i, j)] * c.scale[i] * c.scale[j]; }
    if (!c.reuse_diagonal)
      for (int j = 0; j < 6; ++j) c.diagonal[j] = fmin(fmax(Hs[hidx(j, j)], 1e-6), 1e32);  // min/max_lm_diagonal
    for (int j = 0; j < 6; ++j) D2[j] = c.diagonal[j] / c.radius;
    double y[6];
    const bool ok = chol_solve6(Hs, D2, gs, y);
    c.reuse_diagonal = 1;
    bool valid = false;
    double step[6];
    if (ok) {
      double sg = 0.0, shs = 0.0;
      for (int i = 0; i < 6; ++i) step[i] = -y[i];
      for (int i = 0; i < 6; ++i) {
        sg += step[i] * gs[i];
        for (int j = 0; j < 6; ++j) shs += step[i] * step[j] * Hs[i <= j ? hidx(i, j) : hidx(j, i)];
      }
      c.model_cost_change = -sg - 0.5 * shs;  // -(J step)'(r + J step / 2)
      valid = c.model_cost_change > 0.0;
    }
    if (!valid) {  // HandleInvalidStep
      if (++c.num_invalid >= 5) return lm_done(c, 5);
      c.radius *= 0.5; c.reuse_diagonal = 1; c.step_is_successful = 0;
      continue;
    }
    c.num_invalid = 0;
    double delta[6];
    for (int j = 0; j < 6; ++j) delta[j] = step[j] * c.scale[j];
    state_plus(c.x, delta, c.xc);
    c.action = 1;
    return;
  }
}

__device__ void lm_after_jacobian(LmCtrl& c, const double* acc) {
  for (int k = 0; k < 21; ++k) c.H[k] = acc[k];
  for (int k = 0; k < 6; ++k) c.g[k] = acc[21 + k];
  c.x_cost = acc[27];
  c.sum.jac_evals++;
  if (c.first) {
    c.sum.num_residual_blocks = (int)(acc[28] + 0.5);
    c.sum.initial_cost = c.x_cost;
    for (int j = 0; j < 6; ++j) c.scale[j] = 1.0 / (1.0 + sqrt(c.H[hidx(j, j)]));  // jacobi_scaling, once
    double s = 0.0; for (int k = 0; k < 7; ++k) s += c.x[k] * c.x[k];
    c.x_norm = sqrt(s);
    c.step_is_successful = 1; c.iteration = 0; c.first = 0;
    if (c.sum.num_residual_blocks == 0) return lm_done(c, 4);
  }
  double ng[6], xp[7];
  for (int j = 0; j < 6; ++j) ng[j] = -c.g[j];
  state_plus(c.x, ng, xp);
  double mx = 0.0; for (int k = 0; k < 7; ++k) mx = fmax(mx, fabs(xp[k] - c.x[k]));
  c.gradient_max_norm = mx;
  lm_try_step(c);
}

// `acc` holds cost AND normal equations at the candidate xc: the Jacobian is evaluated in the same pass
// as the cost (speculating on acceptance, which is the common case), so an accepted step needs no
// second pass over the residual blocks.  Rejected steps simply discard it.  The counters keep Ceres'
// meaning (a Jacobian evaluation is counted only when the step is accepted).
__device__ void lm_after_cost(LmCtrl& c, const double* acc) {
  double candidate_cost = acc[27];
  c.sum.cost_evals++;
  if (!isfinite(candidate_cost)) candidate_cost = c.x_cost;
  double sn = 0.0; for (int k = 0; k < 7; ++k) sn += (c.x[k] - c.xc[k]) * (c.x[k] - c.xc[k]);
  if (sqrt(sn) <= 1e-8 * (c.x_norm + 1e-8)) return lm_done(c, 2);                 // parameter_tolerance
  const double cost_change = c.x_cost - candidate_cost;
  if (fabs(cost_change) <= 1e-6 * c.x_cost) return lm_done(c, 3);                 // function_tolerance
  const double rel = cost_change / c.model_cost_change;
  if (rel > 1e-3) {  // HandleSuccessfulStep
    for (int k = 0; k < 7; ++k) c.x[k] = c.xc[k];
    double s = 0.0; for (int k = 0; k < 7; ++k) s += c.x[k] * c.x[k];
    c.x_norm = sqrt(s);
    c.sum.successful_steps++;
    const double u = 2.0 * rel - 1.0;
    c.radius = fmin(1e16, c.radius / fmax(1.0 / 3.0, 1.0 - u * u * u));
    c.decrease_factor = 2.0; c.reuse_diagonal = 0; c.step_is_successful = 1;
    lm_after_jacobian(c, acc);   // gradient / Jacobian at the new point, then the next trust-region step
    return;
  }
  c.step_is_successful = 0;  // HandleUnsuccessfulStep
  c.radius = c.radius / c.decrease_factor; c.decrease_factor *= 2.0; c.reuse_diagonal = 1;
  lm_try_step(c);
}

// Residual and tangent Jacobian of Point2LineFactor (include/liodom/factors.hpp:71-105),
// analytic form of what ceres autodiff + EigenQuaternionParameterization produce
// (SURVEY.md App. A.4): d lp / d delta = -2 [R c]x, d lp / d t = I,
// d w / d t = ((c-t)_x, (c-t)_y, 0) / (rho * (max-min)).
template <bool JAC>
__device__ __forceinline__ void eval_block(const double* cab, const double* x, double min_d, double inv_range, double* acc) {
  const double cx = cab[0], cy = cab[1], cz = cab[2];
  const double qx = x[0], qy = x[1], qz = x[2], qw = x[3];
  // Eigen q*v: uv = 2 qv x v ; v + w uv + qv x uv
  double ux = 2.0 * (qy * cz - qz * cy), uy = 2.0 * (qz * cx - qx * cz), uz = 2.0 * (qx * cy - qy * cx);
  const double rx = cx + qw * ux + (qy * uz - qz * uy), ry = cy + qw * uy + (qz * ux - qx * uz), rz = cz + qw * uz + (qx * uy - qy * ux);
  const double lx = rx + x[4], ly = ry + x[5], lz = rz + x[6];
  const double ax = lx - cab[3], ay = ly - cab[4], az = lz - cab[5];
  const double bx = lx - cab[6], by = ly - cab[7], bz = lz - cab[8];
  const double nx = ay * bz - az * by, ny = az * bx - ax * bz, nz = ax * by - ay * bx;
  const double dex = cab[3] - cab[6], dey = cab[4] - cab[7], dez = cab[5] - cab[8];
  const double inv_den = 1.0 / sqrt(dex * dex + dey * dey + dez * dez);
  const double px = cx - x[4], py = cy - x[5];
  const double rho = sqrt(px * px + py * py);
  const double w = 1.01 - (rho - min_d) * inv_range;
  const double r0 = w * (nx * inv_den), r1 = w * (ny * inv_den), r2 = w * (nz * inv_den);
  const double s = r0 * r0 + r1 * r1 + r2 * r2;
  double rho0, rho1;
  if (s > 0.04) { const double r = sqrt(s); rho0 = 0.4 * r - 0.04; rho1 = fmax(DBL_MIN, 0.2 / r); }
  else { rho0 = s; rho1 = 1.0; }
  acc[27] += 0.5 * rho0;
  acc[28] += 1.0;
  if (JAC) {
    const double sc = sqrt(rho1);
    const double wd = w * inv_den * sc;
    double J[3][6];
    // rotation columns: dlp_k = 2 e_k x u (u = R c), dnu_k = dlp_k x de
    const double u0 = rx, u1 = ry, u2 = rz;
    const double dl[3][3] = {{0.0, -2.0 * u2, 2.0 * u1}, {2.0 * u2, 0.0, -2.0 * u0}, {-2.0 * u1, 2.0 * u0, 0.0}};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double vx = dl[k][0], vy = dl[k][1], vz = dl[k][2];
      J[0][k] = wd * (vy * dez - vz * dey);
      J[1][k] = wd * (vz * dex - vx * dez);
      J[2][k] = wd * (vx * dey - vy * dex);
    }
    // translation columns: w (e_k x de)/den + (nu/den) dw/dt_k
    const double dwx = rho > 0.0 ? px / rho * inv_range : 0.0, dwy = rho > 0.0 ? py / rho * inv_range : 0.0;
    const double n0 = nx * inv_den * sc, n1 = ny * inv_den * sc, n2 = nz * inv_den * sc;
    J[0][3] = n0 * dwx;             J[1][3] = wd * (-dez) + n1 * dwx; J[2][3] = wd * dey + n2 * dwx;
    J[0][4] = wd * dez + n0 * dwy;  J[1][4] = n1 * dwy;               J[2][4] = wd * (-dex) + n2 * dwy;
    J[0][5] = wd * (-dey);          J[1][5] = wd * dex;               J[2][5] = 0.0;
    const double c0 = sc * r0, c1 = sc * r1, c2 = sc * r2;
    int h = 0;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
#pragma unroll
      for (int j = i; j < 6; ++j) { acc[h] += J[0][i] * J[0][j] + J[1][i] * J[1][j] + J[2][i] * J[2][j]; ++h; }
      acc[21 + i] += J[0][i] * c0 + J[1][i] * c1 + J[2][i] * c2;
    }
  }
}

// Deterministic CTA reduction of `count` doubles per thread: warp shuffle tree, then the
// per-warp partials are summed in warp order by the first `count` threads.
template <int first, int count>
__device__ __forceinline__ void block_reduce(double* acc, double* sred /*[warps][kNumAcc]*/, double* out) {
  const int ln = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int k = first; k < first + count; ++k) {
    double v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (ln == 0) sred[w * kNumAcc + k] = v;
  }
  __syncthreads();
  if ((int)threadIdx.x >= first && (int)threadIdx.x < first + count) {
    double s = 0.0;
    for (int ww = 0; ww < nw; ++ww) s += sred[ww * kNumAcc + threadIdx.x];
    out[threadIdx.x] = s;
  }
  __syncthreads();
}

// Result of a solve -> LaserOdometer state: param_q / param_t, odom_ rebuilt from them without
// renormalising (src/laser_odometry.cc:222-227), solver summary.
__device__ void solve_commit(const DevBuffers& d, int lane_b, int outer_it, LmCtrl& c) {
  OdomState& os = d.ostate[lane_b];
  c.sum.iterations = c.iteration;
  c.sum.final_cost = c.x_cost;
  for (int k = 0; k < 4; ++k) os.q[k] = c.x[k];
  for (int k = 0; k < 3; ++k) os.t[k] = c.x[4 + k];
  const double x = c.x[0], y = c.x[1], z = c.x[2], w = c.x[3];
  const double tx = 2 * x, ty = 2 * y, tz = 2 * z;
  const double twx = tx * w, twy = ty * w, twz = tz * w, txx = tx * x, txy = ty * x, txz = tz * x, tyy = ty * y, tyz = tz * y, tzz = tz * z;
  os.odom[0] = 1 - (tyy + tzz); os.odom[1] = txy - twz; os.odom[2] = txz + twy; os.odom[3] = c.x[4];
  os.odom[4] = txy + twz; os.odom[5] = 1 - (txx + tzz); os.odom[6] = tyz - twx; os.odom[7] = c.x[5];
  os.odom[8] = txz - twy; os.odom[9] = tyz + twx; os.odom[10] = 1 - (txx + tyy); os.odom[11] = c.x[6];
  d.diag[lane_b].solve[outer_it] = c.sum;
}

__device__ void lm_init(LmCtrl& c, const OdomState& os) {
  for (int k = 0; k < 4; ++k) c.x[k] = os.q[k];
  for (int k = 0; k < 3; ++k) c.x[4 + k] = os.t[k];
  c.radius = 1e4; c.decrease_factor = 2.0; c.reuse_diagonal = 0; c.num_invalid = 0; c.first = 1; c.action = 0;
  c.iteration = 0; c.step_is_successful = 1;
  SolveSummaryDev z = {}; c.sum = z;
}

// One thread-block CLUSTER per lane runs the whole solve.  The residual blocks are strided over
// the cluster's CTAs; every evaluation ends in a fixed-order reduction (warp shuffle tree ->
// warps in order -> CTAs in rank order through distributed shared memory), so the result does
// not depend on scheduling.  CTA 0 / thread 0 is the trust-region controller; its decision
// (next point + action) is read back by the other CTAs through DSMEM.
// F32: residual blocks come from k_associate (float records {c,a,b,valid}); otherwise from a
// caller-provided double array (liodom_solve, tests).
// OCC = CTAs per SM the register budget is compiled for: 1 (≈200 registers, no spills: lowest latency, used for
// small batches) or 2 (128 registers with spills: two clusters' worth of warps per SM, 20 % faster at 128 lanes).
template <bool F32, int OCC>
__global__ void __launch_bounds__(kSolveThreads, OCC) k_solve(DevBuffers d, int lane0, int outer_it, const double* cab_in, int n_in,
                                                          double* qt_inout, SolveSummaryDev* sum_out) {
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned C = cluster.num_blocks(), crank = cluster.block_rank();
  const DevParams& p = d.p;
  const int lane_b = lane_at(d, lane0 + (int)(blockIdx.x / C));
  OdomState& os = d.ostate[lane_b];
  if (F32 && !os.init) return;   // uniform over the cluster
  __shared__ LmCtrl c;                                         // authoritative copy lives in CTA 0
  __shared__ double sred[(kSolveThreads / 32) * kNumAcc];
  __shared__ double total[kNumAcc];                            // this CTA's partial sums
  __shared__ double ctot[kNumAcc];                             // cluster totals (CTA 0)
  __shared__ double bx[8];                                     // evaluation point + action, local copy
  const int n = F32 ? os.n_edges : n_in;
  const float* blocks = d.blocks + (size_t)lane_b * p.Ecap * 10;
  const double min_d = p.min_range, inv_range = 1.0 / (p.max_range - p.min_range);
  if (crank == 0 && threadIdx.x == 0) {
    lm_init(c, os);
    if (!F32) for (int k = 0; k < 7; ++k) c.x[k] = qt_inout[k];
  }
  // Compact the residual blocks this CTA owns (a contiguous share of the edge list) into a list of the VALID ones:
  // only ~half of the edges pass the line gate, and skipping them inside the evaluation loop left 18 of 32 threads
  // busy per instruction (profiles/step_r02z_lanes128.txt).  Stable (edge order), so the sums stay deterministic.
  __shared__ unsigned short vlist[kValidCap];
  __shared__ int wcnt[kSolveThreads / 32 + 1];
  __shared__ int nvalid_s;
  const int per = (n + (int)C - 1) / (int)C;
  const int share0 = (int)crank * per, share1 = min(n, share0 + per);
  const bool compact = F32 && per <= kValidCap && n <= 65535;
  if (compact) {
    const int ln = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int base = 0;
    for (int i0 = share0; i0 < share1; i0 += blockDim.x) {
      const int i = i0 + (int)threadIdx.x;
      const bool ok = i < share1 && blocks[(size_t)i * 10 + 9] != 0.0f;
      const unsigned m = __ballot_sync(0xffffffffu, ok);
      if (ln == 0) wcnt[w] = __popc(m);
      __syncthreads();
      int off = base;
      for (int ww = 0; ww < w; ++ww) off += wcnt[ww];
      if (ok) vlist[off + __popc(m & ((1u << ln) - 1u))] = (unsigned short)i;
      for (int ww = 0; ww < nw; ++ww) base += wcnt[ww];
      __syncthreads();
    }
    if (threadIdx.x == 0) nvalid_s = base;
    __syncthreads();
  }
  const LmCtrl* lead = cluster.map_shared_rank(&c, 0);
  for (;;) {
    cluster.sync();   // the controller's decision is visible
    if (threadIdx.x < 8) {
      const int action = lead->action;
      bx[threadIdx.x] = threadIdx.x < 7 ? (action == 0 ? lead->x[threadIdx.x] : lead->xc[threadIdx.x]) : (double)action;
    }
    __syncthreads();
    const int action = (int)bx[7];
    if (action == 2) break;
    double xs[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) xs[k] = bx[k];
    double acc[kNumAcc];
#pragma unroll
    for (int k = 0; k < kNumAcc; ++k) acc[k] = 0.0;
    if (compact) {
      const int nv = nvalid_s;
      for (int j = threadIdx.x; j < nv; j += blockDim.x) {
        const float* b = blocks + (size_t)vlist[j] * 10;
        double cab[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) cab[k] = (double)b[k];
        eval_block<true>(cab, xs, min_d, inv_range, acc);   // cost and Jacobian in one pass (see lm_after_cost)
      }
    } else
    for (int i = (int)crank * blockDim.x + threadIdx.x; i < n; i += (int)C * blockDim.x) {
      double cab[9];
      if (F32) {
        const float* b = blocks + (size_t)i * 10;
        if (b[9] == 0.0f) continue;
#pragma unroll
        for (int k = 0; k < 9; ++k) cab[k] = (double)b[k];
      } else {
#pragma unroll
        for (int k = 0; k < 9; ++k) cab[k] = cab_in[(size_t)i * 9 + k];
      }
      eval_block<true>(cab, xs, min_d, inv_range, acc);   // cost and Jacobian in one pass (see lm_after_cost)
    }
    block_reduce<0, kNumAcc>(acc, sred, total);
    cluster.sync();   // every CTA's partials are ready
    if (crank == 0) {
      if ((int)threadIdx.x < kNumAcc) {
        double s = 0.0;
        for (unsigned r = 0; r < C; ++r) s += cluster.map_shared_rank(total, r)[threadIdx.x];
        ctot[threadIdx.x] = s;
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        if (action == 0) lm_after_jacobian(c, ctot);
        else lm_after_cost(c, ctot);
      }
    }
  }
  if (crank == 0 && threadIdx.x == 0) {
    if (F32) solve_commit(d, lane_b, outer_it, c);
    else {
      c.sum.iterations = c.iteration;
      c.sum.final_cost = c.x_cost;
      for (int k = 0; k < 7; ++k) qt_inout[k] = c.x[k];
      if (sum_out) *sum_out = c.sum;
    }
  }
  cluster.sync();   // nobody leaves while its shared memory may still be read
}

// Cluster size: as many CTAs per lane as keep the whole grid in one wave (148 SMs x `occ` resident
// 256-thread CTAs per SM).
static int solve_cluster_size(int nlanes, int occ) {
  int c = 8;
  while (c > 1 && nlanes * c > 148 * occ) c >>= 1;
  return c;
}

template <bool F32>
static void launch_solve_kernel(const DevBuffers& d, cudaStream_t s, int lane0, int nlanes, int outer_it, const double* cab, int n,
                                double* qt, SolveSummaryDev* sum) {
  const int occ = nlanes >= 16 ? 2 : 1;   // measured: the 2-per-SM build wins from 32 lanes up, loses 8 % on a single lane
  const int C = solve_cluster_size(nlanes, occ);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(nlanes * C));
  cfg.blockDim = dim3(kSolveThreads);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  if (occ == 2) cudaLaunchKernelEx(&cfg, k_solve<F32, 2>, d, lane0, outer_it, cab, n, qt, sum);
  else cudaLaunchKernelEx(&cfg, k_solve<F32, 1>, d, lane0, outer_it, cab, n, qt, sum);
}

// ---- point-sharded solve: evaluation over this rank's edges, all-reduce, replicated controller ----
// One kernel per LM evaluation, kShardCtas CTAs: every CTA's thread 0 first advances the trust-region controller from
// the all-reduced sums of the previous evaluation (redundantly and identically: the state is double-buffered, CTA 0
// publishes the new copy), then the CTAs evaluate this rank's share of the residual blocks at the controller's next
// point; partial sums go to global memory and the last CTA to arrive adds them in CTA order (deterministic) into
// the buffer the all-reduce works on.  Per solve: 6 launches + 5 ncclAllReduce(29 x f64).
constexpr int kShardThreads = 256;
constexpr int kShardCtas = 16;
constexpr int kShardMaxEvals = 5;   // the initial evaluation + one (cost + Jacobian) evaluation per iteration (<= 4)

struct ShardState {
  LmCtrl c[2];
  double partial[kShardCtas][32];
  unsigned ticket;
};

size_t shard_ctrl_bytes() { return sizeof(ShardState); }

__global__ void __launch_bounds__(kShardThreads) k_shard_step(DevBuffers d, int lane_b, int rank, int world, int e, int outer_it) {
  const DevParams& p = d.p;
  ShardState& st = static_cast<ShardState*>(d.shard_ctrl)[lane_b];
  const OdomState& os = d.ostate[lane_b];
  __shared__ LmCtrl c;
  __shared__ double sred[(kShardThreads / 32) * kNumAcc];
  __shared__ double total[kNumAcc];
  __shared__ int s_last;
  const int tid = threadIdx.x;
  if (tid == 0) {
    if (e == 0) {
      lm_init(c, os);
      if (!os.init) c.action = 2;   // first frame: no solve
    } else {
      c = st.c[e & 1];
      const double* acc = d.shard_acc + (size_t)lane_b * 32;
      if (c.action == 0) lm_after_jacobian(c, acc);
      else if (c.action == 1) lm_after_cost(c, acc);
    }
    if (blockIdx.x == 0) st.c[(e + 1) & 1] = c;
  }
  __syncthreads();
  if (e == kShardMaxEvals) {   // the controller has seen every evaluation: commit
    if (blockIdx.x == 0 && tid == 0 && os.init) {
      solve_commit(d, lane_b, outer_it, c);
      d.diag[lane_b].n_matches[outer_it] = c.sum.num_residual_blocks;   // all ranks' matches (from the reduced count)
    }
    return;
  }
  const int action = c.action;
  double acc[kNumAcc];
#pragma unroll
  for (int k = 0; k < kNumAcc; ++k) acc[k] = 0.0;
  if (action != 2) {
    double xs[7];
    for (int k = 0; k < 7; ++k) xs[k] = action == 0 ? c.x[k] : c.xc[k];
    const int E = os.n_edges;
    const int share = edge_share(E, world);
    const int t1 = min(E, (rank + 1) * share);
    const float* blocks = d.blocks + (size_t)lane_b * p.Ecap * 10;
    const int* perm = d.perm + (size_t)lane_b * p.Ecap;
    const double min_d = p.min_range, inv_range = 1.0 / (p.max_range - p.min_range);
    for (int t = rank * share + blockIdx.x * kShardThreads + tid; t < t1; t += gridDim.x * kShardThreads) {
      const float* b = blocks + (size_t)perm[t] * 10;
      if (b[9] == 0.0f) continue;
      double cab[9];
#pragma unroll
      for (int k = 0; k < 9; ++k) cab[k] = (double)b[k];
      eval_block<true>(cab, xs, min_d, inv_range, acc);
    }
  }
  block_reduce<0, kNumAcc>(acc, sred, total);
  if (tid < kNumAcc) st.partial[blockIdx.x][tid] = total[tid];
  __threadfence();
  __syncthreads();
  if (tid == 0) s_last = (atomicAdd(&st.ticket, 1u) == gridDim.x - 1) ? 1 : 0;
  __syncthreads();
  if (s_last) {   // every CTA's partials are visible: add them in CTA order
    __threadfence();
    if (tid < kNumAcc) {
      double sum = 0.0;
      for (unsigned b = 0; b < gridDim.x; ++b) sum += ((volatile double*)st.partial[b])[tid];
      d.shard_acc[(size_t)lane_b * 32 + tid] = sum;
    }
    if (tid == 0) st.ticket = 0u;
  }
}

int launch_solve_shard(const DevBuffers& d, cudaStream_t s, int lane, int outer_it, const ShardComm* sc, int* nccl_rc) {
  int k = 0;
  for (int e = 0; e <= kShardMaxEvals; ++e) {
    k_shard_step<<<kShardCtas, kShardThreads, 0, s>>>(d, lane, sc->rank, sc->world, e, outer_it); ++k;
    if (e < kShardMaxEvals) {
      const int rc = shard_allreduce_f64(sc, d.shard_acc + (size_t)lane * 32, kNumAcc, s);
      if (rc != 0 && nccl_rc) *nccl_rc = rc;
    }
  }
  return k;
}

int launch_solve(const DevBuffers& d, cudaStream_t s, LaneRange lr, int outer_it) {
  launch_solve_kernel<true>(d, s, lr.lane0, lr.nlanes, outer_it, nullptr, 0, nullptr, nullptr);
  return 1;
}

int launch_solve_blocks(const DevBuffers& d, cudaStream_t s, int lane, const double* cab, int n, double* qt_inout, SolveSummaryDev* sum) {
  launch_solve_kernel<false>(d, s, lane, 1, 0, cab, n, qt_inout, sum);
  return 1;
}

}  // namespace liodom
