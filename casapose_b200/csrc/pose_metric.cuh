// K8 — ADD / ADD-S / 2-D reprojection errors of a batch of poses (SURVEY.md section 8f-3).
//
// Stands in for map_estimates + evaluate_poses
// (/root/reference/casapose/pose_estimation/ransac_voting.py:561-625, 628-687), which the reference runs as a
// serial tf.map_fn over (image, class): project the evaluation points with the estimated and the ground-truth
// pose (project_tf, :173-182, float32), mean 2-D distance, mean 3-D distance (ADD) or — for the two symmetric
// LINEMOD meshes, recognised by their vertex counts 7862 / 3417 (:618) — the mean closest-point distance
// (ADD-S), which the reference takes from the float64 expansion |a|^2 - 2ab + |b|^2 over all N x N pairs
// (:596-610).  Here the N x N search runs on the float32 points as the direct squared difference
// (a-b).(a-b) — no cancellation, relative error 2e-7 of the squared distance, against the expansion's absolute
// error of about 1e-10 mm^2: both far inside the 1e-5 relative tolerance of the parity test — because FP32 issues
// four times faster than FP64 on this part.
//
//   k_pose_project  one block per object: guards, both projections, err_2d, ADD; symmetric objects leave their
//                   two point clouds (float32 xyz) in scratch;
//   k_adds_min      (256-row tile, object stride): every thread owns one ground-truth point and scans the estimated
//                   cloud through shared memory — FP32-issue-bound, 7 instructions per pair;
//   k_pose_finalize sums the tile partials in order, applies the 0.1*diameter and 2-D thresholds.
// Output rows are map_estimates' own: [err_2d, err_3d, valid_3d, valid_2d, missing, false_positive].
#pragma once
#include "common.cuh"

namespace casa {

constexpr int kMetricThreads = 256;
constexpr int kAddsTile = 1024;  // estimated points per shared-memory pass
constexpr int kAddsGridY = 65535;  // gridDim.y limit: k_adds_min strides over objects beyond it

struct PoseErrParams {
  int n, m, maxp;
  float allowed_2d;
};

__device__ __forceinline__ bool adds_symmetric(int count) { return count == 7862 || count == 3417; }  // :618

// sequential float32 sum of the 12 pose entries (tf.reduce_sum(pose), :575-579)
__device__ __forceinline__ float pose_sum(const float* p) {
  float s = 0.f;
  for (int k = 0; k < 12; ++k) s = __fadd_rn(s, p[k]);
  return s;
}

// project_tf (:173-182): xyz @ R^T + t, then @ K^T, xy / z  — float32, one rounding per op
__device__ __forceinline__ void project_point(const float* P, const float* RT, const float* K, float2& uv, float3& c) {
  c.x = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(P[0], RT[0]), __fmul_rn(P[1], RT[1])), __fmul_rn(P[2], RT[2])), RT[3]);
  c.y = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(P[0], RT[4]), __fmul_rn(P[1], RT[5])), __fmul_rn(P[2], RT[6])), RT[7]);
  c.z = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(P[0], RT[8]), __fmul_rn(P[1], RT[9])), __fmul_rn(P[2], RT[10])), RT[11]);
  const float u = __fadd_rn(__fadd_rn(__fmul_rn(c.x, K[0]), __fmul_rn(c.y, K[1])), __fmul_rn(c.z, K[2]));
  const float v = __fadd_rn(__fadd_rn(__fmul_rn(c.x, K[3]), __fmul_rn(c.y, K[4])), __fmul_rn(c.z, K[5]));
  const float w = __fadd_rn(__fadd_rn(__fmul_rn(c.x, K[6]), __fmul_rn(c.y, K[7])), __fmul_rn(c.z, K[8]));
  uv.x = __fdiv_rn(u, w);
  uv.y = __fdiv_rn(v, w);
}

__device__ __forceinline__ double block_sum(double v, double* sh) {  // fixed order: deterministic
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if (lane == 0) sh[wid] = v;
  __syncthreads();
  double s = 0;
  if (threadIdx.x == 0)
    for (int k = 0; k < kMetricThreads / 32; ++k) s += sh[k];
  __syncthreads();
  return s;  // valid in thread 0
}

// state[obj]: 0 = row already final, 1 = ADD done (err in base), 2 = ADD-S pending
__global__ void __launch_bounds__(kMetricThreads)
    k_pose_project(PoseErrParams pp, const float* __restrict__ poses, const float* __restrict__ poses_gt,
                   const float* __restrict__ cam, const float* __restrict__ model_pts, const int* __restrict__ model_cnt,
                   const int* __restrict__ obj_model, const int* __restrict__ valid, float4* __restrict__ cloud_gt,
                   float4* __restrict__ cloud_est, float* __restrict__ base, int* __restrict__ state, float* __restrict__ out) {
  __shared__ double sh[kMetricThreads / 32];
  __shared__ float sRT[12], sGT[12], sK[9];
  const int obj = blockIdx.x;
  if (threadIdx.x < 12) {
    sRT[threadIdx.x] = poses[(size_t)obj * 12 + threadIdx.x];
    sGT[threadIdx.x] = poses_gt[(size_t)obj * 12 + threadIdx.x];
  }
  if (threadIdx.x < 9) sK[threadIdx.x] = cam[(size_t)obj * 9 + threadIdx.x];
  __syncthreads();
  const float psum = pose_sum(sRT);
  float* row = out + (size_t)obj * 6;
  if (valid[obj] == 0) {  // :573-576
    if (threadIdx.x < 6) row[threadIdx.x] = (threadIdx.x == 5 && fabsf(psum) > 0.0001f) ? 1.f : 0.f;
    if (threadIdx.x == 0) state[obj] = 0;
    return;
  }
  if (fabsf(psum) < 0.0001f) {  // :577-578 object could not be found at all
    if (threadIdx.x == 0) {
      row[0] = 99.9f; row[1] = 999.9f; row[2] = 0.f; row[3] = 0.f; row[4] = 1.f; row[5] = 0.f;
      state[obj] = 0;
    }
    return;
  }
  const int model = obj_model ? obj_model[obj] : obj % pp.m;
  const int cnt = min(model_cnt[model], pp.maxp);
  const bool sym = adds_symmetric(cnt) && cloud_gt != nullptr;
  const float* pts = model_pts + (size_t)model * pp.maxp * 3;
  double e2 = 0, e3 = 0;
  for (int i = threadIdx.x; i < cnt; i += kMetricThreads) {
    float2 ue, ug;
    float3 ce, cg;
    project_point(pts + 3 * i, sRT, sK, ue, ce);
    project_point(pts + 3 * i, sGT, sK, ug, cg);
    const float dx = __fsub_rn(ug.x, ue.x), dy = __fsub_rn(ug.y, ue.y);
    e2 += (double)__fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));  // tf.norm(axis=1), :591
    if (sym) {
      cloud_gt[(size_t)obj * pp.maxp + i] = make_float4(cg.x, cg.y, cg.z, 0.f);
      cloud_est[(size_t)obj * pp.maxp + i] = make_float4(ce.x, ce.y, ce.z, 0.f);
    } else {
      const float a = __fsub_rn(cg.x, ce.x), b = __fsub_rn(cg.y, ce.y), c = __fsub_rn(cg.z, ce.z);
      e3 += (double)__fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b)), __fmul_rn(c, c)));  // :621
    }
  }
  e2 = block_sum(e2, sh);
  e3 = block_sum(e3, sh);
  if (threadIdx.x == 0) {
    base[2 * obj] = (float)(e2 / cnt);
    base[2 * obj + 1] = (float)(e3 / cnt);
    state[obj] = sym ? 2 : 1;
  }
}

// grid (tiles, min(n, kAddsGridY)): rows = ground-truth points, scan = estimated points (adds_error(target, estimate),
// :619).  Objects stride over blockIdx.y, so the object count is not bound by the 65535 limit of gridDim.y; partial
// sums are indexed [obj][tile] with `tiles` row tiles per object.
__global__ void __launch_bounds__(kMetricThreads)
    k_adds_min(PoseErrParams pp, int tiles, const int* __restrict__ model_cnt, const int* __restrict__ obj_model,
               const int* __restrict__ state, const float4* __restrict__ cloud_gt, const float4* __restrict__ cloud_est,
               double* __restrict__ partial) {
  __shared__ float4 sB[kAddsTile];
  __shared__ double sh[kMetricThreads / 32];
  for (int obj = blockIdx.y; obj < pp.n; obj += gridDim.y) {  // uniform per block: the barriers below stay uniform
    if (state[obj] != 2) continue;
    const int model = obj_model ? obj_model[obj] : obj % pp.m;
    const int cnt = min(model_cnt[model], pp.maxp);
    const int row0 = blockIdx.x * kMetricThreads;
    if (row0 >= cnt) continue;
    const int r = row0 + threadIdx.x;
    const float4 a = cloud_gt[(size_t)obj * pp.maxp + min(r, cnt - 1)];
    const float4* B = cloud_est + (size_t)obj * pp.maxp;
    float best0 = INFINITY, best1 = INFINITY;  // two chains: the minimum is exact in any order
    for (int t0 = 0; t0 < cnt; t0 += kAddsTile) {
      const int nt = min(kAddsTile, cnt - t0);
      __syncthreads();
      for (int k = threadIdx.x; k < nt; k += kMetricThreads) sB[k] = B[t0 + k];
      __syncthreads();
      int k = 0;
#pragma unroll 4
      for (; k + 1 < nt; k += 2) {
        const float4 b0 = sB[k], b1 = sB[k + 1];
        const float x0 = a.x - b0.x, y0 = a.y - b0.y, z0 = a.z - b0.z;
        const float x1 = a.x - b1.x, y1 = a.y - b1.y, z1 = a.z - b1.z;
        best0 = fminf(best0, fmaf(x0, x0, fmaf(y0, y0, z0 * z0)));
        best1 = fminf(best1, fmaf(x1, x1, fmaf(y1, y1, z1 * z1)));
      }
      if (k < nt) {
        const float4 b0 = sB[k];
        const float x0 = a.x - b0.x, y0 = a.y - b0.y, z0 = a.z - b0.z;
        best0 = fminf(best0, fmaf(x0, x0, fmaf(y0, y0, z0 * z0)));
      }
    }
    const double best = (double)fminf(best0, best1);
    const double v = r < cnt ? (double)(float)sqrt(fabs(best) + 1e-5) : 0.0;  // :609, cast to float32 per point
    const double s = block_sum(v, sh);
    if (threadIdx.x == 0) partial[(size_t)obj * tiles + blockIdx.x] = s;
  }
}

__global__ void k_pose_finalize(PoseErrParams pp, int tiles, const int* __restrict__ model_cnt, const int* __restrict__ obj_model,
                                const int* __restrict__ state, const float* __restrict__ base, const double* __restrict__ partial,
                                const float* __restrict__ diameters, float* __restrict__ out) {
  const int obj = blockIdx.x * blockDim.x + threadIdx.x;
  if (obj >= pp.n || state[obj] == 0) return;
  const int model = obj_model ? obj_model[obj] : obj % pp.m;
  const int cnt = min(model_cnt[model], pp.maxp);
  float e3 = base[2 * obj + 1];
  if (state[obj] == 2) {
    double s = 0;
    const int used = (cnt + kMetricThreads - 1) / kMetricThreads;
    for (int t = 0; t < used && t < tiles; ++t) s += partial[(size_t)obj * tiles + t];
    e3 = (float)(s / cnt);
  }
  const float e2 = base[2 * obj];
  float* row = out + (size_t)obj * 6;
  row[0] = e2;
  row[1] = e3;
  row[2] = e3 < __fmul_rn(diameters[obj], 0.1f) ? 1.f : 0.f;  // :623
  row[3] = e2 < pp.allowed_2d ? 1.f : 0.f;                     // :624
  row[4] = 0.f;
  row[5] = 0.f;
}

}  // namespace casa
