// K2-K4 — the RANSAC loop of ransac_voting_batch
// (/root/reference/casapose/pose_estimation/ransac_voting.py:310-368) for every (image, class) job.
//
//   k_hypgen     idxs -> hypotheses, exact float32 sequence (:319-322, :197-227), classifies each
//                hypothesis for the filtered predicate and zeroes the vote counters
//   k_plan       loop state of every job (:310-316, round 0) and the exclusive prefixes of scoring work
//                items / refinement tiles over the jobs
//   k_score      THE HOT KERNEL: hypotheses x pixels inlier test (:230-249) and vote counts (:327)
//   k_update     arg-max per keypoint (:328-333), best-so-far update (:336-338), stop test (:340-347)
//   k_refine_solve  re-vote of the winners, normal-equation sums (:349-362); the job's last block applies the
//                invertibility test and the 2x2 solve (:254-272, :364-368)
#pragma once
#include "common.cuh"
#include "philox.cuh"
#include "predicate.cuh"

namespace casa {

// Directions come from the compacted buffer written by k_gather_dirs: `vd` points at the array of one
// (job, keypoint), indexed by the pixel's position t in the job's list.  Stored (dy, dx) like the network
// output; returned as (dx, dy) like tf.reverse(..., axis=[2]) at :308.
__device__ __forceinline__ float2 load_dir(const float2* __restrict__ vd, int t) {
  const float2 s = __ldg(vd + t);
  return make_float2(s.y, s.x);
}

__device__ __forceinline__ const float2* job_dirs(const WS& ws, const Dims& d, int img, int job, int tn, int v) {
  return ws.vdir + ((size_t)img * d.cap + ws.job_off[job]) * d.vn + (size_t)v * tn;
}

// ------------------------------------------------------------------------------------ K2
// grid (ceil(hn*vn/256), J): one thread per (keypoint, hypothesis) of an active job, hypotheses fastest — the three
// [J][vn][hn] outputs are written in full lines (hypothesis-fastest threads wrote them with a stride of hn entries)
__global__ void __launch_bounds__(256) k_hypgen(WS ws, Dims d, FilterConsts fc, const int32_t* __restrict__ idxs, int rnd,
                                                float* dbg_hyps) {
  const int job = blockIdx.y;
  if (!(ws.job_flags[job] & JOB_ACTIVE)) return;
  if (rnd < 0) rnd = ws.ctrl[CTRL_ROUND];  // inside the device-driven loop (rounds >= 1)
  const int e = blockIdx.x * 256 + threadIdx.x;
  if (e >= d.hn * d.vn) return;
  const int tn = ws.job_tn[job];
  const int img = job / d.oc, cls = job - img * d.oc;
  const uint32_t* pix = ws.pix + (size_t)img * d.cap + ws.job_off[job];
  const int v = e / d.hn, h = e - v * d.hn;
  const float2* vd = job_dirs(ws, d, img, job, tn, v);
  int2 ip;
  if (idxs) {
    const int32_t* src = idxs + ((((size_t)job * d.max_iter + rnd) * d.hn + h) * d.vn + v) * 2;
    ip = make_int2(src[0], src[1]);
    if ((unsigned)ip.x >= (unsigned)tn || (unsigned)ip.y >= (unsigned)tn) {
      atomicOr(reinterpret_cast<unsigned*>(&ws.ctrl[CTRL_STATUS]), CASA_STATUS_IDX_RANGE);
      ip.x = min(max(ip.x, 0), tn - 1);
      ip.y = min(max(ip.y, 0), tn - 1);
    }
  } else {
    ip = philox_idx_pair((uint32_t)h, (uint32_t)v, (uint32_t)d.vn, (uint32_t)rnd, (uint32_t)cls,
                         (uint32_t)(d.image_offset + img), (uint32_t)tn, d.seed_lo, d.seed_hi);
  }
  const uint32_t p0 = pix[ip.x], p1 = pix[ip.y];
  const int x0 = p0 & 0xFFFFu, y0 = p0 >> 16, x1 = p1 & 0xFFFFu, y1 = p1 >> 16;
  const float2 c0 = make_float2((float)x0 + 0.5f, (float)y0 + 0.5f);  // :306
  const float2 c1 = make_float2((float)x1 + 0.5f, (float)y1 + 0.5f);
  const float2 d0 = load_dir(vd, ip.x);
  const float2 d1 = load_dir(vd, ip.y);
  const float2 hp = exact_hypothesis(c0, c1, d0, d1);
  const size_t o = ((size_t)job * d.vn + v) * d.hn + h;
  ws.hyp_true[o] = hp;
  const int kind = classify_hypothesis(hp.x, hp.y, fc.fast_ok != 0);
  const float qnan = __int_as_float(0x7fc00000);
  ws.hyp_filt[o] = kind == 0 ? hp : make_float2(qnan, qnan);
  if (kind == 2) {
    const int slot = atomicAdd(&ws.n_exact[job * d.vn + v], 1);
    ws.exact_list[((size_t)job * d.vn + v) * d.hn + slot] = h;
    atomicAdd(&ws.stats[2], 1ull);
  }
  ws.counts[o] = 0;
  if (dbg_hyps) {
    float* dst = dbg_hyps + ((((size_t)job * d.max_iter + rnd) * d.hn + h) * d.vn + v) * 2;
    dst[0] = hp.x;
    dst[1] = hp.y;
  }
}

// ------------------------------------------------------------------------------------ plan
// single block (any multiple of 32 threads up to 1024): item_start[j] = sum over active jobs j' < j of ceil(tn/128) * vn;  (round 0 only)
// rtile_start[j] = sum over live jobs of ceil(tn/1024)
__global__ void __launch_bounds__(1024) k_plan(WS ws, Dims d, int rnd) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (rnd < 0) rnd = ws.ctrl[CTRL_ROUND];  // inside the device-driven loop (rounds >= 1)
  __shared__ int swarp[2][32];
  __shared__ int srun[2];
  if (tid < 2) srun[tid] = 0;
  __syncthreads();
  for (int s = 0; s < d.J; s += (int)blockDim.x) {
    const int job = s + tid;
    int ci = 0, cr = 0;
    if (job < d.J) {
      const int flags = ws.job_flags[job];  // JOB_ACTIVE and the best-so-far state of round 0 come from k_place
      const int tn = ws.job_tn[job];
      if (flags & JOB_ACTIVE) ci = ((tn + kChunk - 1) / kChunk) * d.vn;
      if (!(flags & JOB_GATED) && tn > 0) cr = (tn + d.rtile - 1) / d.rtile;
    }
    int xi = ci, xr = cr;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int yi = __shfl_up_sync(0xffffffffu, xi, o), yr = __shfl_up_sync(0xffffffffu, xr, o);
      if (lane >= o) {
        xi += yi;
        xr += yr;
      }
    }
    if (lane == 31) {
      swarp[0][warp] = xi;
      swarp[1][warp] = xr;
    }
    __syncthreads();
    int wi = 0, wr = 0;
    for (int k = 0; k < warp; ++k) {
      wi += swarp[0][k];
      wr += swarp[1][k];
    }
    const int ri = srun[0], rr = srun[1];
    if (job < d.J) {
      ws.item_start[job] = ri + wi + xi - ci;
      if (rnd == 0) {
        const int r0 = rr + wr + xr - cr;
        ws.rtile_start[job] = r0;
        const int4 rec = make_int4(job, 0, ws.job_tn[job], ws.job_off[job]);
        for (int k = 0; k < cr; ++k) {
          ws.rtile_job[r0 + k] = job;
          ws.rtile_rec[r0 + k] = make_int4(rec.x, k, rec.z, rec.w);
        }
      }
    }
    __syncthreads();
    if (tid == (int)blockDim.x - 1) {
      srun[0] = ri + wi + xi;
      srun[1] = rr + wr + xr;
    }
    __syncthreads();
  }
  if (tid == 0) {
    ws.item_start[d.J] = srun[0];
    ws.ctrl[CTRL_NITEMS] = srun[0];
    ws.ctrl[CTRL_WORK] = 0;
    ws.ctrl[CTRL_NACTIVE] = 0;
    if (rnd == 0) {
      ws.rtile_start[d.J] = srun[1];
      ws.ctrl[CTRL_NRTILES] = srun[1];
    }
  }
}

// ------------------------------------------------------------------------------------ K3
struct ScoreArgs {
  WS ws;
  Dims d;
  FilterConsts fc;
  unsigned one;  // 1, opaque to the compiler: keeps the sign accumulation an IMAD (FMA pipe) instead of an ALU-pipe add
};

// 0xFFFF in the low / high half of the result if a / b has its sign bit set (PRMT with sign-replicating selectors).
__device__ __forceinline__ unsigned prmt_sign2(float a, float b) {
  unsigned r;
  asm("prmt.b32 %0, %1, %2, 0xFFBB;" : "=r"(r) : "r"(__float_as_uint(a)), "r"(__float_as_uint(b)));
  return r;
}

// Tuning constants of k_score, chosen by same-box A/B builds (profiles/r02_ab.txt).  The kernel is bound by dispatch
// cycles, and the register allocation ptxas finds for the 440-instruction loop body moves the result by +-2 %:
//   hypotheses per lane 8 (16: 128 registers, -8..-13 %), TWO resident blocks/SM at 113 registers (the kernel keeps its
//   rate down to two blocks per SM — it is bound by issue slots, not occupancy — and without the 64-register squeeze
//   ptxas finds a schedule of the same 434-instruction loop that runs 2.2 % faster: 0.709 against 0.726 ms; 4 blocks at
//   64 registers was the form of the first half of round 2, 3 at 80: -2 %; register caps of 72..120 through
//   __maxnreg__ or a larger launch-bounds thread count: all slower, 0.723..0.783 ms), 8 pixels per trip (16: the same,
//   4: -1 %), binary search over item_start (a 16-byte record per chunk removed the search but cost 2-4 % through a
//   worse allocation of the loop).
constexpr int kHypPerLaneWide = 8;    // hypotheses (and private counters) per lane of a scoring warp
constexpr int kHypPerLaneNarrow = 4;  // second instantiation for small hypothesis counts (see score_hpl())
constexpr int kScoreMinBlocks = 2;    // resident 256-thread blocks per SM the kernel is compiled for
constexpr int kPixUnroll = 8;         // pixels per trip of the scoring loop

// Exact inlier count of one hypothesis over pixels [t0, t0+npx) of a job, whole warp cooperating.
__device__ __noinline__ int exact_count(const uint32_t* __restrict__ pix, const float2* __restrict__ vd, int t0, int npx,
                                        float hx, float hy, float thr) {
  const int lane = threadIdx.x & 31;
  int c = 0;
  for (int q = lane; q < npx; q += 32) {
    const uint32_t pk = pix[t0 + q];
    const int x = pk & 0xFFFFu, y = pk >> 16;
    const float2 dv = load_dir(vd, t0 + q);
    c += exact_inlier(hx, hy, (float)x + 0.5f, (float)y + 0.5f, dv.x, dv.y, exact_norm(dv.x, dv.y), thr) ? 1 : 0;
  }
  return __reduce_add_sync(0xffffffffu, c);
}

// Stage 2 of the filter for the two hypotheses (a, b) of a flagged pair: every lane re-evaluates its
// pixels of the chunk from the shared-memory coefficients with the per-unit band
//     |t| < kappa |p| + E        (E = evaluation-error bound of that hypothesis in this chunk)
// and only units inside it are decided by exact_inlier().  Returns the corrections to the two sign
// counts.  A NaN hypothesis (no partner / not a filter hypothesis) never enters the band.
// All kChunk coefficient slots of the chunk are evaluated by one straight-line pass (4 pixels x 2 hypotheses per
// lane, 8 independent FFMA chains, the shared-memory loads issued together; padding slots hold t = +1e30 and never
// enter a band), the in-band units — found by 8 % of the passes — are handled afterwards, and the warp reductions
// run only when some lane has a correction (3 % of the flagged pairs).  The earlier form, a loop over the pixels
// with a branch per iteration, was latency-bound: 9.5 % of the kernel's instructions but
// 28 % of its warp-stall samples (profiles/r01_k_score_source_regions.txt).
__device__ __forceinline__ int2 band_adjust2(const float4* __restrict__ cA, const float2* __restrict__ cB, int qb, int qe,
                                             float ax, float ay, float bx, float by, float ea, float eb, float kappa2,
                                             const float2* __restrict__ hfilt, int ha, int hb_ok,
                                             const uint32_t* __restrict__ pix, const float2* __restrict__ vd, int t0,
                                             float thr, unsigned& n_exact) {
  const int lane = threadIdx.x & 31;
  unsigned inband = 0u;  // bit 2k: hypothesis a at pixel slot k*32+lane, bit 2k+1: hypothesis b
#pragma unroll
  for (int k = 0; k < kChunk / 32; ++k) {
    const float4 A = cA[k * 32 + lane];
    const float2 B = cB[k * 32 + lane];
    float pa, pb;
    const float ta = local_unit(A, B, ax, ay, pa);
    const float tb = local_unit(A, B, bx, by, pb);
    inband |= (fabsf(ta) < fmaf(kappa2, fabsf(pa), ea) ? 1u : 0u) << (2 * k);
    inband |= (fabsf(tb) < fmaf(kappa2, fabsf(pb), eb) ? 1u : 0u) << (2 * k + 1);
  }
  if (!hb_ok) inband &= 0x55555555u;
  int da = 0, db = 0;
  if (inband) {  // ~1e-5 of the units
#pragma unroll 1
    for (int k = 0; k < kChunk / 32; ++k) {
      const unsigned two = (inband >> (2 * k)) & 3u;
      const int q = k * 32 + lane;
      if (two == 0u || q < qb || q >= qe) continue;
      const float4 A = cA[q];  // same instructions on the same operands as above: the same t, bit for bit
      const float2 B = cB[q];
      float pa, pb;
      const float ta = local_unit(A, B, ax, ay, pa);
      const float tb = local_unit(A, B, bx, by, pb);
      const uint32_t pk = pix[t0 + q];
      const int x = pk & 0xFFFFu, y = pk >> 16;
      const float2 dv = load_dir(vd, t0 + q);
      const float nd = exact_norm(dv.x, dv.y);
      if (two & 1u) {
        const float2 h = hfilt[ha];
        da += (exact_inlier(h.x, h.y, (float)x + 0.5f, (float)y + 0.5f, dv.x, dv.y, nd, thr) ? 1 : 0) -
              (int)(__float_as_uint(ta) >> 31);
      }
      if (two & 2u) {
        const float2 h = hfilt[ha + 32];
        db += (exact_inlier(h.x, h.y, (float)x + 0.5f, (float)y + 0.5f, dv.x, dv.y, nd, thr) ? 1 : 0) -
              (int)(__float_as_uint(tb) >> 31);
      }
      n_exact += __popc(two);
    }
  }
  if (!__any_sync(0xffffffffu, (da | db) != 0)) return make_int2(0, 0);
  return make_int2(__reduce_add_sync(0xffffffffu, da), __reduce_add_sync(0xffffffffu, db));
}

// K3 — THE HOT KERNEL.  Persistent grid of independent warps; each warp pulls (job, keypoint,
// 128-pixel chunk) items from a global counter.  No block barriers.
//
//  * chunk-local coordinates: o = centre of the chunk's bounding box, c' = c - o (exact, one
//    fractional bit), h' = fl(h - o) once per (hypothesis, chunk);
//  * per pixel 6 coefficients in warp-private shared memory (24 B, broadcast LDS.128 + LDS.64):
//        p = D hy' - E hx' - P0          (= d^ x (h - c))
//        s = A0 - G hx' - H hy'          (= -k d^ . (h - c),  k = tan(theta0))
//        t = |p| + s                     inlier <=> sign(t)
//    5 FP32-pipe instructions per unit; the sign bits of a hypothesis pair are turned into two 16-bit fields by one
//    PRMT and accumulated by one IMAD (FMA pipe) — every negative unit adds 0xFFFF to its field, decoded after the
//    chunk — i.e. 1/2 PRMT + 1/2 IMAD + 1/2 FMNMX3 per unit (the LEA.HI per unit of the first version cost two
//    dispatch cycles: profiles/r02_loop_bench.txt);
//  * every lane owns 8 hypotheses and their private counters (no shuffles/ballots/atomics in the loop);
//  * min |t| per hypothesis pair is compared with B = c1 (|h'| + R): if min|t| >= B every sign in the
//    chunk is provably the reference's verdict (predicate.cuh / DESIGN.md); otherwise band_adjust()
//    finds the (rare) units that need the exact predicate.
//  * a warp sweeps the hypotheses in groups of 32 * kHypPerLane; the kernel is instantiated for 8 (groups of 256) and
//    for 4 hypotheses per lane (groups of 128: twice the shared-memory loads per unit, but a round of 128 hypotheses —
//    BASELINE config 5's smallest sweep point — fills its group instead of half of it).
template <int kHypPerLane>
__global__ void __launch_bounds__(kScoreThreads, kScoreMinBlocks) k_score(ScoreArgs a) {
  __shared__ float4 sA[kScoreWarps][kChunk];  // (D, -E, -P0, A0)
  __shared__ float2 sB[kScoreWarps][kChunk];  // (-G, -H)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int hn = a.d.hn;
  const int n_items = a.ws.ctrl[CTRL_NITEMS];
  const int n_groups = (hn + 32 * kHypPerLane - 1) / (32 * kHypPerLane);
  const int n_full = max(0, n_items - (int)(gridDim.x * kScoreWarps));  // items before the split tail
  const int n_virtual = n_full + (n_items - n_full) * n_groups;
  float4* cA = sA[warp];
  float2* cB = sB[warp];
  const float qnan = __int_as_float(0x7fc00000);
  unsigned n_exact = 0u, n_flagged = 0u;  // per-lane diagnostics, flushed once when the warp leaves
  for (;;) {
    int item = 0;
    if (lane == 0) item = atomicAdd(&a.ws.ctrl[CTRL_WORK], 1);
    item = __shfl_sync(0xffffffffu, item, 0);
    if (item >= n_virtual) break;
    // The last `n_items - n_full` items are handed out one hypothesis group at a time, so that the tail of the
    // persistent grid is a group (half an item at 512 hypotheses) instead of an item.  (Splitting the pixels of the
    // tail items as well made the main loop's range variable and the whole kernel 1.7 % slower: profiles/r02_ab.txt.)
    int g_begin = 0, g_end = n_groups;
    if (item >= n_full) {
      const int j = item - n_full;
      item = n_full + j / n_groups;
      g_begin = j - (j / n_groups) * n_groups;
      g_end = g_begin + 1;
    }
    // item -> (job, chunk, keypoint): binary search in the per-job prefix of work items
    int lo = 0, hi = a.d.J;
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (__ldg(&a.ws.item_start[mid]) <= item) lo = mid; else hi = mid;
    }
    const int job = lo;
    const int rem = item - __ldg(&a.ws.item_start[job]);
    const int chunk = rem / a.d.vn, v = rem - chunk * a.d.vn;
    const int img = job / a.d.oc;
    const int tn = a.ws.job_tn[job];
    const uint32_t* pix = a.ws.pix + (size_t)img * a.d.cap + a.ws.job_off[job];
    const float2* vd = job_dirs(a.ws, a.d, img, job, tn, v);
    const int t0 = chunk * kChunk;
    const int npx = min(kChunk, tn - t0);
    const bool first_part = g_begin == 0;  // the exact list and the exact whole-chunk path run once per item

    // pixels of the chunk (4 per lane), bounding box, origin
    int px[kChunk / 32], py[kChunk / 32];
    float2 dvs[kChunk / 32];
    int xmin = 0x7fffffff, xmax = 0, ymin = 0x7fffffff, ymax = 0;
#pragma unroll
    for (int k = 0; k < kChunk / 32; ++k) {
      const int q = k * 32 + lane;
      px[k] = py[k] = -1;
      dvs[k] = make_float2(0.f, 0.f);
      if (q < npx) {
        const uint32_t pk = pix[t0 + q];
        px[k] = pk & 0xFFFFu;
        py[k] = pk >> 16;
        dvs[k] = load_dir(vd, t0 + q);
        xmin = min(xmin, px[k]); xmax = max(xmax, px[k]);
        ymin = min(ymin, py[k]); ymax = max(ymax, py[k]);
      }
    }
    xmin = __reduce_min_sync(0xffffffffu, xmin); xmax = __reduce_max_sync(0xffffffffu, xmax);
    ymin = __reduce_min_sync(0xffffffffu, ymin); ymax = __reduce_max_sync(0xffffffffu, ymax);
    const float ox = 0.5f * (float)(xmin + xmax) + 0.5f;  // exact: at most one fractional bit
    const float oy = 0.5f * (float)(ymin + ymax) + 0.5f;

    __syncwarp();  // previous item's readers are done with cA / cB
    bool weird = false;
    float rr = 0.f;
#pragma unroll
    for (int k = 0; k < kChunk / 32; ++k) {
      const int q = k * 32 + lane;
      float4 A = make_float4(0.f, 0.f, 0.f, 1.0e30f);  // invalid / padding pixel: t = +1e30, never inlier, never flagged
      float2 B = make_float2(0.f, 0.f);
      if (px[k] >= 0) {
        const float cxl = ((float)px[k] + 0.5f) - ox, cyl = ((float)py[k] + 0.5f) - oy;  // c' = c - o, exact
        rr = fmaxf(rr, oct_norm(cxl, cyl));
        weird |= !make_local_coef(cxl, cyl, dvs[k].x, dvs[k].y, a.fc.k_mid, A, B);
      }
      cA[q] = A;
      cB[q] = B;
    }
    rr = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(rr)));  // non-negative floats order like uints
    weird = __any_sync(0xffffffffu, weird);
    __syncwarp();

    const size_t hoff = ((size_t)job * a.d.vn + v) * hn;
    int* gc = a.ws.counts + hoff;
    const float2* htrue = a.ws.hyp_true + hoff;
    if (a.fc.fast_ok == 0 || weird) {  // rare: whole chunk with the exact predicate
      if (!first_part) continue;
      for (int h = 0; h < hn; ++h) {
        const float2 hp = htrue[h];
        const int c = exact_count(pix, vd, t0, npx, hp.x, hp.y, a.fc.thr);
        if (lane == 0 && c) atomicAdd(&gc[h], c);
      }
      if (a.ws.stats && lane == 0) atomicAdd(&a.ws.stats[1], (unsigned long long)npx * hn);
      continue;
    }

    const float2* hfilt = a.ws.hyp_filt + hoff;
    for (int g = g_begin; g < g_end; ++g) {
      float hx[kHypPerLane], hy[kHypPerLane], mn[kHypPerLane / 2];
      unsigned acc[kHypPerLane / 2];  // two 16-bit sign counters per hypothesis pair (a 128-pixel chunk cannot overflow them)
#pragma unroll
      for (int i = 0; i < kHypPerLane; ++i) {
        const int h = (g * kHypPerLane + i) * 32 + lane;
        float2 hp = make_float2(qnan, qnan);
        if (h < hn) hp = hfilt[h];
        hx[i] = hp.x - ox;  // h' = fl(h - o)
        hy[i] = hp.y - oy;
      }
#pragma unroll
      for (int i = 0; i < kHypPerLane / 2; ++i) {
        mn[i] = 3.0e38f;
        acc[i] = 0u;
      }
#pragma unroll(kPixUnroll)
      for (int q = 0; q < npx; ++q) {
        const float4 A = cA[q];
        const float2 B = cB[q];
#pragma unroll
        for (int i = 0; i < kHypPerLane; i += 2) {
          float p0, p1;
          const float t0v = local_unit(A, B, hx[i], hy[i], p0);
          const float t1v = local_unit(A, B, hx[i + 1], hy[i + 1], p1);
          acc[i >> 1] = prmt_sign2(t0v, t1v) * a.one + acc[i >> 1];
          mn[i >> 1] = fminf(fminf(mn[i >> 1], fabsf(t0v)), fabsf(t1v));
        }
      }
      unsigned nlo[kHypPerLane];
#pragma unroll
      for (int i = 0; i < kHypPerLane; i += 2) {  // acc = 0xFFFF n_lo + 0xFFFF0000 n_hi  (mod 2^32)
        nlo[i] = (0u - acc[i >> 1]) & 0xFFFFu;
        nlo[i + 1] = (nlo[i] - ((acc[i >> 1] + nlo[i]) >> 16)) & 0xFFFFu;
      }
      // pairs whose closest unit is inside the uncertainty bound (NaN compares false)
      unsigned flagged = 0u;
#pragma unroll
      for (int i = 0; i < kHypPerLane; i += 2) {
        const float nmax = fmaxf(oct_norm(hx[i], hy[i]), oct_norm(hx[i + 1], hy[i + 1])) + rr;
        flagged |= (mn[i >> 1] < a.fc.c1 * nmax ? 1u : 0u) << (i >> 1);
      }
#pragma unroll
      for (int i = 0; i < kHypPerLane; ++i) {
        const int h = (g * kHypPerLane + i) * 32 + lane;
        if (h < hn && nlo[i]) atomicAdd(&gc[h], (int)nlo[i]);
      }
      // stage 2, after the group's registers are dead: corrections go straight to the global counters
      if (__any_sync(0xffffffffu, flagged != 0u)) {
        for (int i2 = 0; i2 < kHypPerLane / 2; ++i2) {
          unsigned m = __ballot_sync(0xffffffffu, (flagged >> i2) & 1u);
          while (m) {
            const int src = __ffs(m) - 1;
            m &= m - 1;
            const int ha = (g * kHypPerLane + 2 * i2) * 32 + src;
            const bool hb_ok = ha + 32 < hn;
            const float2 pa = hfilt[ha];
            const float2 pb = hb_ok ? hfilt[ha + 32] : make_float2(qnan, qnan);
            const float ax = pa.x - ox, ay = pa.y - oy, bx = pb.x - ox, by = pb.y - oy;  // same h' as the main loop
            const float ea = a.fc.e1 * (oct_norm(ax, ay) + rr), eb = a.fc.e1 * (oct_norm(bx, by) + rr);
            const int2 dd = band_adjust2(cA, cB, 0, npx, ax, ay, bx, by, ea, eb, a.fc.kappa2, hfilt, ha, hb_ok, pix, vd,
                                         t0, a.fc.thr, n_exact);
            if (lane == 0) {
              if (dd.x) atomicAdd(&gc[ha], dd.x);
              if (dd.y) atomicAdd(&gc[ha + 32], dd.y);
              ++n_flagged;
            }
          }
        }
      }
    }
    // hypotheses the filter cannot take (exact list)
    const int nlist = first_part ? a.ws.n_exact[job * a.d.vn + v] : 0;
    for (int k = 0; k < nlist; ++k) {
      const int h = a.ws.exact_list[hoff + k];
      const float2 hp = htrue[h];
      const int c = exact_count(pix, vd, t0, npx, hp.x, hp.y, a.fc.thr);
      if (lane == 0 && c) atomicAdd(&gc[h], c);
    }
  }
  if (a.ws.stats) {
    n_exact = __reduce_add_sync(0xffffffffu, n_exact);
    if (lane == 0 && n_exact) atomicAdd(&a.ws.stats[1], (unsigned long long)n_exact);
    if (lane == 0 && n_flagged) atomicAdd(&a.ws.stats[3], (unsigned long long)n_flagged);
  }
}

// Hypotheses per lane for a round of hn hypotheses: the narrow instantiation when the last group of 256 would be at
// most half full (hn mod 256 in 1..128), else the wide one.
inline int score_hpl(int hn) { return ((hn - 1) % (32 * kHypPerLaneWide)) < 32 * kHypPerLaneNarrow ? kHypPerLaneNarrow : kHypPerLaneWide; }

// ------------------------------------------------------------------------------------ stop test
__device__ __forceinline__ double ipow_f64(double x, int n) {  // oracle/ransac_voting_np.py:_ipow_f64
  double r = 1.0, bs = x;
  while (n) {
    if (n & 1) r = __dmul_rn(r, bs);
    bs = __dmul_rn(bs, bs);
    n >>= 1;
  }
  return r;
}

// 1 - (1 - r^2)^hyp_num > confidence   (:344-346, all float32 in the reference)
__device__ __forceinline__ bool stop_test(float min_ratio, int hyp_num, float confidence) {
  const float r2 = __fmul_rn(min_ratio, min_ratio);
  const float base = __fsub_rn(1.0f, r2);
  const float pw = __double2float_rn(ipow_f64((double)base, hyp_num));
  return __fsub_rn(1.0f, pw) > confidence;
}

// ------------------------------------------------------------------------------------ K3b
// one block per job, one warp per keypoint.  The block that finishes last publishes the loop state: the index of the
// next round and — when the call runs as a CUDA graph — the condition of the graph's WHILE node, so that the
// reference's data-dependent `while` (:318) never returns to the host.
__global__ void __launch_bounds__(512) k_update(WS ws, Dims d, int rnd, casa_ransac_debug dbg, unsigned long long cond_handle,
                                                uint32_t* sticky) {
  const int job = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (rnd < 0) rnd = ws.ctrl[CTRL_ROUND];
  const int flags = ws.job_flags[job];
  __shared__ unsigned long long svbest[16];
  if (flags & JOB_ACTIVE) {  // uniform per block
    const int tn = ws.job_tn[job];
    if (warp < d.vn) {
      const int* c = ws.counts + ((size_t)job * d.vn + warp) * d.hn;
      unsigned long long best = 0ull;  // (count << 32) | ~h : max count, then lowest h (:328 argmax takes the first)
      for (int h = lane; h < d.hn; h += 32) {
        const unsigned long long key = ((unsigned long long)(unsigned)c[h] << 32) | (unsigned)(0xFFFFFFFFu - (unsigned)h);
        best = key > best ? key : best;
      }
#pragma unroll
      for (int o = 16; o; o >>= 1) {
        const unsigned long long y = __shfl_xor_sync(0xffffffffu, best, o);
        best = y > best ? y : best;
      }
      if (lane == 0) svbest[warp] = best;
    }
    __syncthreads();
    if (dbg.counts) {
      int32_t* dst = dbg.counts + ((size_t)job * d.max_iter + rnd) * d.hn * d.vn;
      for (int e = tid; e < d.hn * d.vn; e += blockDim.x) {
        const int h = e / d.vn, v = e - h * d.vn;
        dst[e] = ws.counts[((size_t)job * d.vn + v) * d.hn + h];
      }
    }
    if (tid < d.vn) ws.n_exact[job * d.vn + tid] = 0;  // for the next round's k_hypgen
    if (warp == 0) {  // lane v: best-so-far update of keypoint v (:333-338), then the stop test on the minimum (:342-347)
      float best_ratio = 3.0e38f;
      if (lane < d.vn) {
        const int v = lane;
        const int cnt = (int)(svbest[v] >> 32);
        const int widx = (int)(0xFFFFFFFFu - (unsigned)(svbest[v] & 0xFFFFFFFFull));
        const float ratio = __fdiv_rn((float)cnt, (float)tn);  // :333
        best_ratio = ws.win_ratio[job * d.vn + v];
        if (best_ratio < ratio) {                              // :336-338
          best_ratio = ratio;
          ws.win_ratio[job * d.vn + v] = ratio;
          ws.win_pts[job * d.vn + v] = ws.hyp_true[((size_t)job * d.vn + v) * d.hn + widx];
        }
        if (dbg.win_idx) dbg.win_idx[((size_t)job * d.max_iter + rnd) * d.vn + v] = widx;
      }
      float min_ratio = best_ratio;                            // :342 (ratios are non-negative: they order like their bits)
      min_ratio = __uint_as_float(__reduce_min_sync(0xffffffffu, __float_as_uint(min_ratio)));
      if (lane == 0) {
        const int cur_iter = rnd + 1;                            // :341
        const int hyp_num = d.hn * cur_iter;                     // :340 (exact in float32 below 2^24)
        const bool stop = stop_test(min_ratio, hyp_num, d.confidence) || cur_iter >= d.max_iter;  // :344-347
        ws.job_rounds[job] = cur_iter;
        if (stop) {
          ws.job_flags[job] = flags & ~JOB_ACTIVE;
        } else {
          atomicAdd(&ws.ctrl[CTRL_NACTIVE], 1);
        }
        atomicAdd(&ws.stats[0], (unsigned long long)tn * d.vn * d.hn);
      }
    }
  }
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    if (atomicAdd(&ws.ctrl[CTRL_DONE], 1) == (int)gridDim.x - 1) {  // every other block has published its state
      __threadfence();
      const int nactive = *(volatile int*)&ws.ctrl[CTRL_NACTIVE];
      ws.ctrl[CTRL_DONE] = 0;
      ws.ctrl[CTRL_ROUND] = rnd + 1;
      const unsigned st = (unsigned)ws.ctrl[CTRL_STATUS];  // every status bit is raised before or inside the loop
      if (st && sticky) atomicOr(sticky, st);              // -> the handle's sticky word (collected by casa_sync)
      if (cond_handle) cudaGraphSetConditional((cudaGraphConditionalHandle)cond_handle, nactive > 0 ? 1u : 0u);
    }
  }
}

// ------------------------------------------------------------------------------------ K4
// condition number of [[a,b],[b,c]], closed form in float64 (oracle: cond_2x2_sym_f64)
__device__ __forceinline__ bool invertible_2x2(float af, float bf, float cf) {
  const double a = af, b = bf, c = cf;
  const double m = __dmul_rn(__dadd_rn(a, c), 0.5);
  const double dd = __dmul_rn(__dsub_rn(a, c), 0.5);
  const double r = __dsqrt_rn(__dadd_rn(__dmul_rn(dd, dd), __dmul_rn(b, b)));
  double s0 = fabs(__dadd_rn(m, r));
  double s1 = fabs(__dsub_rn(m, r));
  if (s1 > s0) {
    const double t = s0;
    s0 = s1;
    s1 = t;
  }
  if (!(s1 > 0.0)) return false;  // zero or NaN smallest singular value: condition number inf / nan
  const double cnd = __ddiv_rn(s0, s1);
  return isfinite(cnd) && cnd < 1000000.0;  // :270-272, eps_inv = float32(1/1e-6)
}

constexpr int kRefineThreads = 256;

// lane u of one warp: sums of keypoint u -> invertibility (:364, all-or-nothing), solve (:367), outputs of the job
__device__ __forceinline__ void solve_job(const WS& ws, const Dims& d, int job, bool dead, const float (&q)[5], bool inv,
                                          float* __restrict__ out, const casa_ransac_debug& dbg) {
  const int u = threadIdx.x & 31;
  const int flags = ws.job_flags[job];
  const int tn = ws.job_tn[job];
  const bool all_inv = !dead && __all_sync(0xffffffffu, inv);  // :364 — one singular keypoint un-refines all
  if (u < d.vn) {
    float2 r = make_float2(0.f, 0.f);  // :291-292
    if (!dead) {
      r = ws.win_pts[job * d.vn + u];  // :364-365
      if (all_inv) {                   // :367  inv(ATA) @ ATb, closed form in float64 on the float32 sums
        const double a = q[0], bq = q[1], c = q[2], g0 = q[3], g1 = q[4];
        const double det = __dsub_rn(__dmul_rn(a, c), __dmul_rn(bq, bq));
        r.x = (float)__ddiv_rn(__dsub_rn(__dmul_rn(c, g0), __dmul_rn(bq, g1)), det);
        r.y = (float)__ddiv_rn(__dsub_rn(__dmul_rn(a, g1), __dmul_rn(bq, g0)), det);
      }
    }
    reinterpret_cast<float2*>(out)[(size_t)job * d.vn + u] = r;
    if (dbg.ata) {
      float* o = dbg.ata + ((size_t)job * d.vn + u) * 3;
      o[0] = q[0]; o[1] = q[1]; o[2] = q[2];
    }
    if (dbg.atb) {
      float* o = dbg.atb + ((size_t)job * d.vn + u) * 2;
      o[0] = q[3]; o[1] = q[4];
    }
    if (dbg.win_pts) reinterpret_cast<float2*>(dbg.win_pts)[(size_t)job * d.vn + u] = dead ? make_float2(0.f, 0.f) : ws.win_pts[job * d.vn + u];
    if (dbg.win_ratio) dbg.win_ratio[(size_t)job * d.vn + u] = dead ? 0.f : ws.win_ratio[job * d.vn + u];
  }
  if (u == 0) {
    if (dbg.refined) dbg.refined[job] = all_inv ? 1 : 0;
    if (dbg.tn0) dbg.tn0[job] = ws.job_tn0[job];
    if (dbg.tn) dbg.tn[job] = (flags & JOB_GATED) ? 0 : tn;
    if (dbg.rounds) dbg.rounds[job] = dead ? 0 : ws.job_rounds[job];
    if (dbg.pix_off) dbg.pix_off[job] = ws.job_off[job];
  }
}

// K4 — refinement and solve.  grid (<= n_rtiles, vn): blocks stride over the (2048-pixel tile of a job, keypoint)
// pairs, 8 pixels per thread (all 16 loads of a thread in flight together).  A block re-votes the winner over its tile (:353) and accumulates the normal equations
// (:356-362): float32 products exactly as the reference forms them (normal * inlier flag, so a non-finite direction
// poisons the sums as it does there), float64 accumulation, fixed reduction order.  The block that finishes a job's
// last (tile, keypoint) pair sums the tiles in order (bit-reproducible), applies the all-or-nothing invertibility
// rule (:364-365) and solves all keypoints of the job (:254-272, :367) — no second kernel.  Jobs without tiles
// (gated, empty) get their zeros from the blocks' first warps.
__global__ void __launch_bounds__(kRefineThreads) k_refine_solve(WS ws, Dims d, FilterConsts fc, float* __restrict__ out,
                                                                 casa_ransac_debug dbg) {
  const int v = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n_rtiles = ws.rtile_start[d.J];
  __shared__ double sred[kRefineThreads / 32][5];
  __shared__ int s_last;
  if (warp == 0 && v == 0) {  // dead jobs: zeros (:291-292) and the debug rows
    for (int job = blockIdx.x; job < d.J; job += gridDim.x) {
      const int tn = ws.job_tn[job];
      if ((ws.job_flags[job] & JOB_GATED) || tn <= 0) {
        const float q[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        solve_job(ws, d, job, true, q, true, out, dbg);
      }
    }
  }
  for (int rt = blockIdx.x; rt < n_rtiles; rt += gridDim.x) {
    const int4 rec = __ldg(&ws.rtile_rec[rt]);  // (job, tile, tn, list offset): one load instead of a chain of three
    const int job = rec.x, tile = rec.y, tn = rec.z;
    const int img = job / d.oc;
    const uint32_t* pix = ws.pix + (size_t)img * d.cap + rec.w;
    const float2* vd = ws.vdir + ((size_t)img * d.cap + rec.w) * d.vn + (size_t)v * tn;
    const float2 wp = ws.win_pts[job * d.vn + v];
    // The re-vote uses the filtered predicate in its direct form (hd = fl(h - c) is the reference's own difference,
    // no chunk origin): t = |d^ x hd| - k d^.hd decides unless |t| < c1 |hd|_1 (c1 >= w + e1 bounds the band and the
    // evaluation error relative to |hd| <= |hd|_1, predicate.cuh; scripts/check_band.py (6)); units inside the band,
    // directions the filter cannot take and winners outside the filter's hypothesis class get the exact sequence.
    // The inlier SET is therefore the reference's, at a quarter of the instructions (IEEE sqrt and divide otherwise).
    const bool fast = fc.fast_ok != 0 && classify_hypothesis(wp.x, wp.y, true) == 0;
    double s[5] = {0, 0, 0, 0, 0};
    // phase 1: all loads of the thread's 4 pixels in flight together; phase 2: arithmetic
    uint32_t lp_[kVoteTile / kRefineThreads];
    float2 ld_[kVoteTile / kRefineThreads];
#pragma unroll
    for (int k = 0; k < kVoteTile / kRefineThreads; ++k) {
      const int t = tile * kVoteTile + k * kRefineThreads + tid;
      lp_[k] = t < tn ? pix[t] : 0u;
      ld_[k] = t < tn ? load_dir(vd, t) : make_float2(0.f, 0.f);
    }
#pragma unroll
    for (int k = 0; k < kVoteTile / kRefineThreads; ++k) {
      const int t = tile * kVoteTile + k * kRefineThreads + tid;
      if (t < tn) {
        const uint32_t pk = lp_[k];
        const int x = pk & 0xFFFFu, y = pk >> 16;
        const float2 dv = ld_[k];
        const float cx = (float)x + 0.5f, cy = (float)y + 0.5f;
        bool in = false, decided = false;
        PixCoef pc;
        if (fast && make_coef(dv.x, dv.y, fc.k_mid, pc)) {
          const float hdx = wp.x - cx, hdy = wp.y - cy;  // the reference's rounded difference (:236)
          const float pv = fmaf(pc.D, hdy, -(pc.E * hdx));
          const float tv = fabsf(pv) - fmaf(pc.G, hdx, pc.H * hdy);
          decided = !(fabsf(tv) < fc.c1 * (fabsf(hdx) + fabsf(hdy)));
          in = (__float_as_uint(tv) >> 31) != 0u;
        }
        if (!decided) in = exact_inlier(wp.x, wp.y, cx, cy, dv.x, dv.y, exact_norm(dv.x, dv.y), fc.thr);  // :353
        const bool finite = fabsf(dv.x) <= 3.0e38f && fabsf(dv.y) <= 3.0e38f;
        if (in || !finite) {  // finite outliers contribute exact zeros
          const float fl = in ? 1.0f : 0.0f;
          const float nx = __fmul_rn(__fmul_rn(dv.y, -1.0f), fl);  // normal = (-dy, dx) * inlier      :349, :356
          const float ny = __fmul_rn(dv.x, fl);
          const float bb = __fadd_rn(__fmul_rn(nx, cx), __fmul_rn(ny, cy));  // :359
          s[0] += (double)__fmul_rn(nx, nx);  // :361
          s[1] += (double)__fmul_rn(nx, ny);
          s[2] += (double)__fmul_rn(ny, ny);
          s[3] += (double)__fmul_rn(nx, bb);  // :362
          s[4] += (double)__fmul_rn(ny, bb);
        }
      }
    }
#pragma unroll
    for (int k = 0; k < 5; ++k) {
#pragma unroll
      for (int o = 16; o; o >>= 1) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
      if (lane == 0) sred[warp][k] = s[k];
    }
    __syncthreads();
    if (tid < 5) {
      double t = 0;
      for (int k = 0; k < kRefineThreads / 32; ++k) t += sred[k][tid];
      ws.partial[((size_t)rt * d.vn + v) * 5 + tid] = t;
    }
    __syncthreads();
    // the block that finishes the job's last (tile, keypoint) pair solves the job
    const int r0 = rt - tile, r1 = r0 + (tn + kVoteTile - 1) / kVoteTile;
    if (tid == 0) {
      __threadfence();
      s_last = atomicAdd(&ws.job_done[job], 1) == (r1 - r0) * d.vn - 1;
    }
    __syncthreads();
    if (s_last && warp == 0) {
      __threadfence();
      float q[5] = {0, 0, 0, 0, 0};
      bool inv = true;
      if (lane < d.vn) {
        double acc[5] = {0, 0, 0, 0, 0};
        for (int r = r0; r < r1; ++r) {  // tiles in order: bit-reproducible sums
          const volatile double* ps = ws.partial + ((size_t)r * d.vn + lane) * 5;
#pragma unroll
          for (int k = 0; k < 5; ++k) acc[k] += ps[k];
        }
#pragma unroll
        for (int k = 0; k < 5; ++k) q[k] = (float)acc[k];  // ATA / ATb are float32 tensors in the reference
        inv = invertible_2x2(q[0], q[1], q[2]);
      }
      solve_job(ws, d, job, false, q, inv, out, dbg);
    }
    __syncthreads();
  }
}

}  // namespace casa
