// K1 — ordered per-class mask compaction.
//
// Replaces  coords = reverse(where(mask != 0)) + 0.5 ; direct = boolean_mask(vertex, mask)
// (/root/reference/casapose/pose_estimation/ransac_voting.py:287-308) for all (image, class)
// pairs of the batch at once:
//   k_mask_bits   reads the mask ONCE (float32, float16 or bfloat16; the only pass over [b,h,w,oc]), writes one
//                 class-membership word per pixel and per-tile class counts (warp ballots);
//   k_place       job table (class offsets, foreground_num gate :290, down-sampling threshold :298), raster-order
//                 scatter of packed pixel coordinates (y<<16 | x) — the order is semantically required because
//                 hypothesis indices address this list (:216) — and the gather of the listed pixels' directions;
//   k_cap_filter  in-place ordered filter  selection < max_num / foreground_num  (:295-301);
//   k_gather_dirs direction gather for what k_place did not take: jobs above max_num (after the filter) and vector
//                 fields in mapped host memory (full-line reads over PCIe).
// Only masked pixels of the 18-channel field are ever read.
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace casa {

// Vectorised path (tile slab 16-byte aligned, i.e. (h*w*oc) % (16 / sizeof(T)) == 0 and an aligned base): the block
// streams its tile's [1024 x oc] elements as one contiguous run of 128-bit loads (4 floats or 8 16-bit values) — every
// warp-load is 512 contiguous bytes, all loads of a thread are independent and in flight together (this matters when
// `mask` is mapped pinned host memory: full-line PCIe reads) — and ORs the few non-zero elements into a shared-memory
// word per pixel.
template <typename T>  // float, __half or __nv_bfloat16
__global__ void __launch_bounds__(256) k_mask_bits(const T* __restrict__ mask, WS ws, Dims d, int vec) {
  constexpr int kPerVec = 16 / sizeof(T);  // elements per 128-bit load
  const int img = blockIdx.y, tile = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31;
  __shared__ int scnt[32];
  __shared__ unsigned sbits[kCountTile];
  if (tid < 32) scnt[tid] = 0;
  const T* mimg = mask + (size_t)img * d.hw * d.oc;
  const int p0 = tile * kCountTile;
  const int npx = min(kCountTile, d.hw - p0);
  bool bad = false;
  uint32_t m[4] = {0u, 0u, 0u, 0u};
  if (vec) {
#pragma unroll
    for (int k = 0; k < 4; ++k) sbits[k * 256 + tid] = 0u;
    __syncthreads();
    const uint4* slab = reinterpret_cast<const uint4*>(mimg + (size_t)p0 * d.oc);
    const int nv = npx * d.oc / kPerVec;  // npx*oc is a multiple of kPerVec on this path
    for (int i0 = 0; i0 < nv; i0 += 256 * 8) {
      uint4 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int i = i0 + u * 256 + tid;
        v[u] = i < nv ? __ldg(slab + i) : make_uint4(0u, 0u, 0u, 0u);
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        // most elements of a one-hot mask are +0: test the four 32-bit words at once (-0 and NaN are non-zero
        // patterns and take the per-element path below)
        if (((v[u].x | v[u].y) | (v[u].z | v[u].w)) == 0u) continue;
        const int e0 = (i0 + u * 256 + tid) * kPerVec;
#pragma unroll
        for (int j = 0; j < kPerVec; ++j) {
          const float f = vec_elem(v[u], j, mask);
          if (f != 0.f) {  // NaN != 0 is true, like tf.not_equal (:304)
            const int e = e0 + j, px = e / d.oc;
            atomicOr(&sbits[px], 1u << (e - px * d.oc));
            bad |= f != 1.f;
          }
        }
      }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) m[k] = sbits[k * 256 + tid];
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int p = p0 + k * 256 + tid;
      if (p < d.hw) {
        const T* row = mimg + (size_t)p * d.oc;
        for (int c = 0; c < d.oc; ++c) {
          const float v = ld_f32(row + c);
          m[k] |= (uint32_t)(v != 0.f) << c;
          bad |= (v != 0.f && v != 1.f);
        }
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int p = p0 + k * 256 + tid;
    if (p < d.hw) ws.bits[(size_t)img * d.hw + p] = m[k];
    if (__any_sync(0xffffffffu, m[k] != 0u)) {
      for (int c = 0; c < d.oc; ++c) {
        const unsigned bal = __ballot_sync(0xffffffffu, (m[k] >> c) & 1u);
        if (lane == 0 && bal) atomicAdd(&scnt[c], __popc(bal));
      }
    }
  }
  if (bad) atomicOr(reinterpret_cast<unsigned*>(&ws.ctrl[CTRL_STATUS]), CASA_STATUS_MASK_NOT_BINARY);
  __syncthreads();
  if (tid < d.oc) ws.tile_cnt[((size_t)img * d.oc + tid) * d.nct + tile] = scnt[tid];
}

// Membership words that were packed on the host (casa_ransac_vote_host): same outputs as k_mask_bits — ws.bits and
// the per-tile class counts — from one u32 per pixel instead of oc floats.
__global__ void __launch_bounds__(256) k_bits_in(const uint32_t* __restrict__ src, WS ws, Dims d, int not_binary) {
  const int img = blockIdx.y, tile = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31;
  __shared__ int scnt[32];
  if (tid < 32) scnt[tid] = 0;
  __syncthreads();
  uint32_t m[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int p = tile * kCountTile + k * 256 + tid;
    m[k] = p < d.hw ? __ldg(src + (size_t)img * d.hw + p) : 0u;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int p = tile * kCountTile + k * 256 + tid;
    if (p < d.hw) ws.bits[(size_t)img * d.hw + p] = m[k];
    if (__any_sync(0xffffffffu, m[k] != 0u)) {
      for (int c = 0; c < d.oc; ++c) {
        const unsigned bal = __ballot_sync(0xffffffffu, (m[k] >> c) & 1u);
        if (lane == 0 && bal) atomicAdd(&scnt[c], __popc(bal));
      }
    }
  }
  if (not_binary && tile == 0 && img == 0 && tid == 0)
    atomicOr(reinterpret_cast<unsigned*>(&ws.ctrl[CTRL_STATUS]), CASA_STATUS_MASK_NOT_BINARY);
  __syncthreads();
  if (tid < d.oc) ws.tile_cnt[((size_t)img * d.oc + tid) * d.nct + tile] = scnt[tid];
}

// Fused pre-step (pose_evaluation.py:36-47): bit c of a pixel is set iff argmax(seg) == c + 1
// (tf.argmax takes the first maximum; NaN scores never win, like Eigen's comparison-based arg-max).
template <typename T>
__global__ void __launch_bounds__(256) k_seg_bits(const T* __restrict__ seg, WS ws, Dims d) {
  const int img = blockIdx.y, tile = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31;
  const int nc = d.oc + 1;
  __shared__ int scnt[32];
  if (tid < 32) scnt[tid] = 0;
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int p = tile * kCountTile + k * 256 + tid;
    uint32_t m = 0;
    if (p < d.hw) {
      const T* row = seg + ((size_t)img * d.hw + p) * nc;
      float best = ld_f32(row);
      int arg = 0;
      for (int c = 1; c < nc; ++c) {
        const float v = ld_f32(row + c);
        if (v > best) {
          best = v;
          arg = c;
        }
      }
      if (arg > 0) m = 1u << (arg - 1);
      ws.bits[(size_t)img * d.hw + p] = m;
    }
    if (__any_sync(0xffffffffu, m != 0u)) {
      for (int c = 0; c < d.oc; ++c) {
        const unsigned bal = __ballot_sync(0xffffffffu, (m >> c) & 1u);
        if (lane == 0 && bal) atomicAdd(&scnt[c], __popc(bal));
      }
    }
  }
  __syncthreads();
  if (tid < d.oc) ws.tile_cnt[((size_t)img * d.oc + tid) * d.nct + tile] = scnt[tid];
}

// Second (and last) pass of the compaction, one block per (1024-pixel tile, image): job table, raster-order scatter
// and — for device-resident vector fields — the direction gather, in one kernel (round 1 and the first half of
// round 2 ran k_job_tables -> k_scatter -> k_gather_dirs: 54 us of launches per 16 frames).
//   * every block that holds a masked pixel re-derives what it needs from the tile counts of its image (oc x nct
//     ints, L2-resident): the class totals = foreground_num (:287) and the totals of the tiles in front of it;
//   * one thread lays out the image's pixel list from the totals: class offsets, the foreground_num gate (:290), the
//     down-sampling threshold (:298), the overflow rule; the block of tile 0 publishes this job table;
//   * masked pixels are written in raster order (ballot + prefix popcount) — semantically required, hypothesis
//     indices address the list (:216) — and, when `gather` is set, the pixel's (dy,dx) row is copied into the
//     keypoint-major direction buffer at the same list position (direct = boolean_mask(vertex, mask), :308).  Jobs
//     above max_num are gathered after k_cap_filter (k_gather_dirs, only_capped), gated jobs never.
constexpr int kPlaceSub = 4;  // count tiles per k_place block (4096 pixels, 16 per thread)
// T: element type of `vertex`; gather requires it aligned to one (dy, dx) pair.
template <int VN, typename T>  // keypoints per row when known at compile time (9), 0 = runtime
__global__ void __launch_bounds__(256, 4) k_place(const T* __restrict__ vertex, WS ws, Dims d, int gather) {
  const int img = blockIdx.y, tile0 = blockIdx.x * kPlaceSub;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kSlots = kPlaceSub * 4;  // pixels per thread; slot j covers pixels [j*256, (j+1)*256) of the block
  __shared__ int wcnt[32][kSlots * 8];   // [class][slot*8 + warp]
  __shared__ int scnt[32], s_tot[32], s_pre[32], s_off[32], s_flags[32];
  // every load the block needs is issued up front (one round trip to L2): its pixels' membership words and the
  // tile counts of its image — warp w scans classes w, w + 8, ...: total, total in front of this block, own count
  uint32_t m[kSlots];
  const int p0 = tile0 * kCountTile;
#pragma unroll
  for (int j = 0; j < kSlots; ++j) {
    const int p = p0 + j * 256 + tid;
    m[j] = p < d.hw ? __ldg(ws.bits + (size_t)img * d.hw + p) : 0u;
  }
  for (int c = warp; c < d.oc; c += 8) {
    const int* cnt = ws.tile_cnt + ((size_t)img * d.oc + c) * d.nct;
    int tot = 0, pre = 0, own = 0;
    for (int t0 = 0; t0 < d.nct; t0 += 320) {  // ten loads per lane in flight (nct = 300 at 480 x 640)
      int v[10];
#pragma unroll
      for (int k = 0; k < 10; ++k) {
        const int t = t0 + k * 32 + lane;
        v[k] = t < d.nct ? __ldg(cnt + t) : 0;
      }
#pragma unroll
      for (int k = 0; k < 10; ++k) {
        const int t = t0 + k * 32 + lane;
        tot += v[k];
        pre += t < tile0 ? v[k] : 0;
        own += (t >= tile0 && t < tile0 + kPlaceSub) ? v[k] : 0;
      }
    }
    tot = __reduce_add_sync(0xffffffffu, tot);
    pre = __reduce_add_sync(0xffffffffu, pre);
    own = __reduce_add_sync(0xffffffffu, own);
    if (lane == 0) {
      s_tot[c] = tot;
      s_pre[c] = pre;
      scnt[c] = own;
    }
  }
  __syncthreads();
  const int mine = tid < d.oc ? scnt[tid] : 0;
  if (__syncthreads_or(mine) == 0 && tile0 != 0) return;  // pure background: nothing to place
  if (tid == 0) {
    int off = 0;
    for (int c = 0; c < d.oc; ++c) {
      const int job = img * d.oc + c;
      const int tn0 = s_tot[c];
      int flags = 0;
      const float fg = (float)tn0;  // tf.reduce_sum of a {0,1} mask (:287)
      if (fg < d.min_num) flags |= JOB_GATED;               // :290
      float thr = 1.f;
      if (fg > d.max_num) {                                 // :295
        flags |= JOB_NEEDS_CAP;
        thr = __fdiv_rn(d.max_num, fg);                     // :298
      }
      if (off + tn0 > d.cap) flags |= JOB_GATED | JOB_OVERFLOW;
      if (!(flags & JOB_GATED) && tn0 > 0) flags |= JOB_ACTIVE;  // loop state of round 0 (:310-316)
      s_off[c] = off;
      s_flags[c] = flags;
      if (tile0 == 0) {
        if (flags & JOB_OVERFLOW) atomicOr(reinterpret_cast<unsigned*>(&ws.ctrl[CTRL_STATUS]), CASA_STATUS_PIX_OVERFLOW);
        ws.job_tn0[job] = tn0;
        ws.job_tn[job] = (flags & JOB_OVERFLOW) ? 0 : tn0;
        ws.job_off[job] = off;
        ws.job_flags[job] = flags;
        ws.job_rounds[job] = 0;
        ws.job_done[job] = 0;
        ws.job_selthr[job] = thr;
      }
      if (!(flags & JOB_OVERFLOW)) off += tn0;
    }
  }
  if (tile0 == 0) {  // best-so-far state of the image's jobs (:310-316); k_hypgen no longer waits for k_plan
    for (int e = tid; e < d.oc * d.vn; e += 256) {
      const size_t o = (size_t)img * d.oc * d.vn + e;
      ws.win_ratio[o] = 0.f;
      ws.win_pts[o] = make_float2(0.f, 0.f);
      ws.n_exact[o] = 0;
    }
  }
  for (int c = 0; c < d.oc; ++c) {
    if (scnt[c] == 0) continue;  // block-uniform
#pragma unroll
    for (int j = 0; j < kSlots; ++j) {
      const unsigned bal = __ballot_sync(0xffffffffu, (m[j] >> c) & 1u);
      if (lane == 0) wcnt[c][j * 8 + warp] = __popc(bal);
    }
  }
  __syncthreads();
  for (int c = warp; c < d.oc; c += 8) {  // exclusive prefix over the class's kSlots*8 warp counts, kPlaceSub per lane
    if (scnt[c] == 0) continue;
    int v[kPlaceSub], tot = 0;
#pragma unroll
    for (int k = 0; k < kPlaceSub; ++k) {
      v[k] = wcnt[c][lane * kPlaceSub + k];
      tot += v[k];
    }
    int x = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    int acc = x - tot;
#pragma unroll
    for (int k = 0; k < kPlaceSub; ++k) {
      wcnt[c][lane * kPlaceSub + k] = acc;
      acc += v[k];
    }
  }
  __syncthreads();
  const int vn = VN ? VN : d.vn;
  const int vslots = vn * d.vpc;
  for (int c = 0; c < d.oc; ++c) {
    if (scnt[c] == 0) continue;
    const int flags = s_flags[c];
    if (flags & JOB_OVERFLOW) continue;
    const int tn = s_tot[c];
    const int tbase = s_pre[c];
    uint32_t* out = ws.pix + (size_t)img * d.cap + s_off[c];
    const bool dirs = gather && !(flags & (JOB_GATED | JOB_NEEDS_CAP));
    using P = typename Pair<T>::type;
    const P* vfield = reinterpret_cast<const P*>(vertex) + (size_t)img * d.hw * vslots + (d.vpc > 1 ? c * vn : 0);
    float2* dst0 = ws.vdir + ((size_t)img * d.cap + s_off[c]) * vn;
#pragma unroll
    for (int j = 0; j < kSlots; ++j) {
      const bool bit = (m[j] >> c) & 1u;
      const unsigned bal = __ballot_sync(0xffffffffu, bit);
      if (bit) {
        const int p = p0 + j * 256 + tid;
        const int y = p / d.w, x = p - y * d.w;
        const int slot = tbase + wcnt[c][j * 8 + warp] + __popc(bal & lanemask_lt());
        out[slot] = ((uint32_t)y << 16) | (uint32_t)x;
        if (dirs) {
          const P* row = vfield + (size_t)p * vslots;
          if (VN) {
            float2 r[VN ? VN : 1];
#pragma unroll
            for (int v = 0; v < VN; ++v) r[v] = ld_pair(row + v);
#pragma unroll
            for (int v = 0; v < VN; ++v) dst0[(size_t)v * tn + slot] = r[v];
          } else {
            for (int v = 0; v < vn; ++v) dst0[(size_t)v * tn + slot] = ld_pair(row + v);
          }
        }
      }
    }
  }
}

// one block of 1024 threads per job; only jobs with JOB_NEEDS_CAP do anything
__global__ void __launch_bounds__(1024) k_cap_filter(WS ws, Dims d, const float* __restrict__ selection) {
  const int job = blockIdx.x;
  const int flags = ws.job_flags[job];
  if (!(flags & JOB_NEEDS_CAP) || (flags & JOB_GATED)) return;
  const int img = job / d.oc, cls = job - img * d.oc;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tn0 = ws.job_tn0[job];
  const float thr = ws.job_selthr[job];
  uint32_t* pix = ws.pix + (size_t)img * d.cap + ws.job_off[job];
  __shared__ int swarp[32];
  __shared__ int srun;
  if (tid == 0) srun = 0;
  __syncthreads();
  for (int s = 0; s < tn0; s += 1024) {
    const int i = s + tid;
    bool keep = false;
    uint32_t pk = 0;
    if (i < tn0) {
      pk = pix[i];
      const int x = pk & 0xFFFFu, y = pk >> 16;
      const float sel = selection ? selection[((size_t)job * d.h + y) * d.w + x]
                                  : philox_selection((uint32_t)(y * d.w + x), (uint32_t)cls,
                                                     (uint32_t)(d.image_offset + img), d.seed_lo, d.seed_hi);
      keep = sel < thr;  // :297-299
    }
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) swarp[warp] = __popc(bal);
    __syncthreads();  // all reads of this chunk are done
    int woff = 0;
    for (int k = 0; k < warp; ++k) woff += swarp[k];
    const int run = srun;
    if (keep) pix[run + woff + __popc(bal & lanemask_lt())] = pk;
    __syncthreads();
    if (tid == 1023) srun = run + woff + __popc(bal);
    __syncthreads();
  }
  if (tid == 0) {
    ws.job_tn[job] = srun;
    if (srun == 0) {
      ws.job_flags[job] = flags & ~JOB_ACTIVE;  // nothing left to vote on (k_place set the flag from foreground_num)
      atomicOr(reinterpret_cast<unsigned*>(&ws.ctrl[CTRL_STATUS]), CASA_STATUS_EMPTY_AFTER_CAP);
    }
  }
}

// Gathers the (dy,dx) vectors of every listed pixel ONCE into the compacted, keypoint-major buffer all
// later kernels read (direct = boolean_mask(vertex, mask), ransac_voting.py:308; for PVNet-style outputs
// the class's own field, pose_evaluation.py:38-45).  One thread per listed pixel: the pixel's 8*vn-byte
// row is read once (the only access to `vertex`, which may be device memory or mapped pinned host
// memory — then only masked pixels of the field cross PCIe), the writes are coalesced per keypoint.
template <int ROWF, typename T>  // elements per pixel row when known at compile time (18 for vn = 9), 0 = runtime
__global__ void __launch_bounds__(256) k_gather_dirs(const T* __restrict__ vertex, WS ws, Dims d, int only_capped) {
  const int job = blockIdx.y, img = job / d.oc, cls = job - img * d.oc;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tn = ws.job_tn[job];
  if (tn <= 0 || (ws.job_flags[job] & JOB_GATED)) return;
  if (only_capped && !(ws.job_flags[job] & JOB_NEEDS_CAP)) return;  // the others were gathered by k_place
  const int vslots = d.vn * d.vpc;
  const int rowf = ROWF ? ROWF : 2 * d.vn;  // elements fetched per pixel (<= 32)
  const T* vfield = vertex + (size_t)img * d.hw * vslots * 2 + (d.vpc > 1 ? cls * d.vn * 2 : 0);
  const int off = ws.job_off[job];
  const uint32_t* pix = ws.pix + (size_t)img * d.cap + off;
  float2* dst0 = ws.vdir + ((size_t)img * d.cap + off) * d.vn;
  __shared__ float srow[8][32][33];  // [warp][pixel][float], padded
  const int nwarps = gridDim.x * 8;
  for (int base = (blockIdx.x * 8 + warp) * 32; base < tn; base += nwarps * 32) {
    const int t = base + lane;  // lane l owns list position base + l
    int px = -1;                // the pixel's index in the image (< 2^30)
    if (t < tn) {
      const uint32_t pk = pix[t];
      px = (int)((pk >> 16) * (uint32_t)d.w + (pk & 0xFFFFu));
    }
    // flattened fetch: element e = lane + 32 k of the warp's [32 pixels x rowf elements] block.  Consecutive
    // lanes read consecutive elements of one row and run on into the next pixel's row, which is contiguous in
    // memory whenever the two pixels are neighbours — so most warp-loads are one full 128-byte line, and all
    // rowf loads of a lane are independent (no per-pixel serialisation).  The row offset px * vn * vpc * 2 is
    // formed in 64 bits: it reaches 2^31 from pixel 2^26 on for a shared field with vn = 16, and from pixel 2^21
    // on for 32 per-class fields with vn = 16.
#pragma unroll 6
    for (int k = 0; k < rowf; ++k) {
      const int e = k * 32 + lane;
      const int src = e / rowf, f = e - src * rowf;
      const int sp = __shfl_sync(0xffffffffu, px, src);
      if (sp >= 0) srow[warp][src][f] = ld_f32(vfield + (size_t)sp * (vslots * 2) + f);
    }
    __syncwarp();
    if (t < tn)
      for (int v = 0; v < d.vn; ++v) dst0[(size_t)v * tn + t] = make_float2(srow[warp][lane][2 * v], srow[warp][lane][2 * v + 1]);
    __syncwarp();
  }
}

}  // namespace casa
