// Shared definitions of the casapose_b200 kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/casapose_b200.h"

namespace casa {

// Element types of the network outputs the input-reading kernels take (casa_dtype): float, __half, __nv_bfloat16.
// Every element is widened exactly to float32 at load; everything after the load is the float32 path, so a 16-bit
// call computes what the float32 call computes on the upcast tensor.
__device__ __forceinline__ float ld_f32(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld_f32(const __half* p) { return __half2float(__ldg(p)); }
__device__ __forceinline__ float ld_f32(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }
// (dy, dx) pairs: Pair<T>::type is the two-element vector of T, ld_pair loads one and widens it
template <typename T> struct Pair;
template <> struct Pair<float> { using type = float2; };
template <> struct Pair<__half> { using type = __half2; };
template <> struct Pair<__nv_bfloat16> { using type = __nv_bfloat162; };
__device__ __forceinline__ float2 ld_pair(const float2* p) { return __ldg(p); }
__device__ __forceinline__ float2 ld_pair(const __half2* p) { return __half22float2(__ldg(p)); }
__device__ __forceinline__ float2 ld_pair(const __nv_bfloat162* p) { return __bfloat1622float2(__ldg(p)); }
// element j of a 16-byte vector holding 16 / sizeof(T) elements of T
__device__ __forceinline__ float vec_elem(const uint4& v, int j, const float*) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
  return __uint_as_float(w[j]);
}
__device__ __forceinline__ float vec_elem(const uint4& v, int j, const __half*) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
  return __half2float(__ushort_as_half((unsigned short)(w[j >> 1] >> (16 * (j & 1)))));
}
__device__ __forceinline__ float vec_elem(const uint4& v, int j, const __nv_bfloat16*) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
  return __uint_as_float((j & 1) ? (w[j >> 1] & 0xFFFF0000u) : (w[j >> 1] << 16));
}

constexpr int kCountTile = 1024;   // pixels per block in the mask / scatter kernels (256 thr x 4)
constexpr int kScoreWarps = 8;     // warps per scoring block
constexpr int kScoreThreads = kScoreWarps * 32;
constexpr int kChunk = 128;        // pixels per scoring work item (one warp); 256: no faster, 64: -5 % (profiles/r02_ab.txt)
constexpr int kRefineTile = 1024;  // pixels per reduction tile of the LS layer (256 threads x 4)
constexpr int kVoteTile = 2048;    // pixels per refinement tile of the voting path (256 threads x 8)

// job flag bits
constexpr int JOB_GATED = 1;     // foreground_num < min_num  -> zeros   (ransac_voting.py:290)
constexpr int JOB_NEEDS_CAP = 2; // foreground_num > max_num             (ransac_voting.py:295)
constexpr int JOB_ACTIVE = 4;    // RANSAC loop still running             (ransac_voting.py:318)
constexpr int JOB_OVERFLOW = 8;  // pixel list did not fit

// ctrl words
constexpr int CTRL_NITEMS = 0;
constexpr int CTRL_WORK = 1;
constexpr int CTRL_NACTIVE = 2;
constexpr int CTRL_STATUS = 3;
constexpr int CTRL_NRTILES = 4;
constexpr int CTRL_ROUND = 5;   // index of the round the loop body is about to run (device-driven loop, rounds >= 1)
constexpr int CTRL_DONE = 6;    // k_update blocks finished in this round (the last one decides about the next round)
constexpr int CTRL_WORDS = 8;

// hypothesis classes written by k_hypgen
//   normal : hyp_filt == hyp_true, scored by the filtered predicate
//   zero   : count is 0 by construction (invalid-sum guard :241-243 or non-finite) -> hyp_filt = NaN
//   exact  : scored only by the exact predicate (exact list)                        -> hyp_filt = NaN

// Constants of the filtered predicate, derived on the host in double (filter_consts()).
struct FilterConsts {
  float thr;     // inlier_thresh as float32
  float k_mid;   // tan(theta0): t = |p| + s changes sign exactly at the threshold angle
  float c1;      // k_score: a chunk's signs are proven if min|t| >= c1 (|h'| + R)
  float e1;      // k_score stage 2: evaluation-error part of the unit band, e1 (|h'| + R)
  float kappa2;  // k_score stage 2: a unit is uncertain only if |t| < kappa2 |p| + e1 (|h'| + R)
  int fast_ok;   // 0 -> thresholds outside the proven range, score everything exactly
};

struct WS {
  uint32_t* bits;      // [b*h*w]        class-membership bit mask per pixel
  int* tile_cnt;       // [b][oc][nct]   per count-tile class counts
  uint32_t* pix;       // [b][cap]       compacted pixel lists, (y<<16|x), raster order per class
  float2* vdir;        // [b][cap*vn]    compacted directions (dy,dx): job j, keypoint v, pixel t at
                       //                (img*cap + job_off[j])*vn + v*tn[j] + t  — gathered once per call
  int* job_tn0;        // [J]
  int* job_tn;         // [J]
  int* job_off;        // [J]
  int* job_flags;      // [J]
  int* job_rounds;     // [J]
  int* job_done;       // [J]            refinement blocks of the job that have finished (the last one solves)
  float* job_selthr;   // [J]            max_num / foreground_num          (:298)
  float* win_ratio;    // [J][vn]
  float2* win_pts;     // [J][vn]
  float2* hyp_true;    // [J][vn][hn]
  float2* hyp_filt;    // [J][vn][hn]
  int* exact_list;     // [J][vn][hn]
  int* n_exact;        // [J][vn]
  int* counts;         // [J][vn][hn]
  int* item_start;     // [J+1]          exclusive prefix of scoring work items (chunks x vn) over active jobs
  int* rtile_start;    // [J+1]          exclusive prefix of refinement tiles over live jobs
  int* rtile_job;      // [max_rtiles]   job of every refinement tile (written by k_plan in round 0)
  int4* rtile_rec;     // [max_rtiles]   (job, tile, tn, list offset) of every refinement tile (k_plan, round 0)
  int* ctrl;           // [CTRL_WORDS]
  double* partial;     // [max(max_rtiles, J)][vn][5]  sums nx*nx, nx*ny, ny*ny, nx*b, ny*b: per (job, keypoint) in the
                       //                voting path, per tile in the LS layer
  unsigned long long* stats;  // [4]
};

struct Dims {
  int b, h, w, oc, vn, hn, max_iter;
  int hw, J, nct, cap, max_rtiles;
  int rtile;  // pixels per refinement tile: kVoteTile (voting) or kRefineTile (LS layer)
  int image_offset;
  uint32_t seed_lo, seed_hi;
  float min_num, max_num, confidence;
  int force_exact;
  int vpc;  // vertex fields per pixel: 1, or oc when every class has its own field
};

__device__ __forceinline__ unsigned lanemask_lt() {
  unsigned m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

}  // namespace casa
