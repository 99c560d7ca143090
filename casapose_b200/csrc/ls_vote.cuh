// K5/K6 — CoordLSVotingWeighted (/root/reference/casapose/pose_estimation/voting_layers_2d.py:5-122).
//
//   k_ls_classify  hot_seg = softmax(1e6 * seg)[..., 1:] (:38-41) per pixel; writes the class-membership
//                  word (hot != 0) for the shared compaction kernels (compaction.cuh) and, for the
//                  component filter, the class whose hot value truncates to 1 (int(hot + 0.1), :44);
//   k_cc_*         4-connected components of all classes at once (union-find on the label map; stands in
//                  for tfa.image.connected_components :53), component sizes, and the reference's selection
//                  bincount -> (<50 -> 0) -> top_k -> index[1] or [2]  (:64-76) including its quirks
//                  (label 0 = background competes; zero counts tie-break towards the lowest label);
//   k_ls_reduce    per (class, keypoint, 1024-pixel tile): n = dir/|dir|, R = w (I - n n^T), q = R p with
//                  p = ((y+.5)/H, (x+.5)/H), weighted by hot (and the component mask); float32 elementwise
//                  exactly as the reference forms them, float64 accumulation (:113-114), fixed order;
//   k_ls_solve     ordered sum of the tiles, 2x2 pseudo-inverse in float64 (:116-120), * height (:122).
// HBM-bound: algorithmic bytes per frame h*w*4*((1+oc) + 2*vn + vn); only masked pixels of the direction
// and confidence fields are actually read (gathered through the pixel lists).
#pragma once
#include "common.cuh"

namespace casa {

constexpr unsigned LS_STATUS_NONFINITE = 16u;  // a non-finite R / q / p (the reference's tf.Assert :109-121)

struct LsDims {
  int b, h, w, nc, oc, vn, hw;
  int sigmoid_weights, filter, which, bins, min_component;
};

struct LsWS {
  unsigned char* cls9;  // [b*hw]  class (1..oc) with int(hot + 0.1) == 1, else 0
  int* parent;          // [b*hw]  union-find forest over same-class 4-neighbours (index inside the image)
  int* count;           // [b*hw]  component size at the root pixel
  int* roots;           // [b*hw]  list of root pixels per image
  int* nroots;          // [b]
  int* sel;             // [J]     selected component: root pixel, -1 = none, -2 = label 0 (background)
  float* wt;            // [b*cap] weight hot * component mask of every listed pixel (job list order)
  float* cconf;         // [b*cap*vn] softplus / sigmoid confidence weights, keypoint-major per job like WS::vdir
  // run-based components (k_cc_runs, forward call): per list entry the index of its horizontal run (-1: not in the
  // class's int mask) and the component mask; run tables in global memory for jobs with more than kCcRuns runs
  int* ridx;            // [b*cap]
  unsigned char* keep;  // [b*cap]
  uint32_t* run_pk;     // [b*cap]  (y << 16 | x0) of the run
  int* run_x1;          // [b*cap]
  int* run_parent;      // [b*cap]
  int* run_cnt;         // [b*cap]
};

constexpr unsigned char kOneHotFlag = 0x80;  // cls9 bit 7 (forward call only): softmax(1e6 seg) is exactly one-hot
constexpr unsigned char kClassMask = 0x3F;

// softmax(seg * 1e6) in float32 (:38-41): z = x * 1e6; e = exp(z - max z); e / sum e
__device__ __forceinline__ void hard_softmax(const float* __restrict__ row, int nc, float* hot) {
  float m = -3.4e38f;
  for (int c = 0; c < nc; ++c) {
    hot[c] = __fmul_rn(__ldg(row + c), 1.0e6f);
    m = fmaxf(m, hot[c]);
  }
  float s = 0.f;
  for (int c = 0; c < nc; ++c) {
    hot[c] = expf(__fsub_rn(hot[c], m));
    s = __fadd_rn(s, hot[c]);
  }
  for (int c = 0; c < nc; ++c) hot[c] = __fdiv_rn(hot[c], s);
}

__device__ __forceinline__ float hard_softmax_one(const float* __restrict__ row, int nc, int cls) {
  float m = -3.4e38f;
  for (int c = 0; c < nc; ++c) m = fmaxf(m, __fmul_rn(__ldg(row + c), 1.0e6f));
  float s = 0.f, e = 0.f;
  for (int c = 0; c < nc; ++c) {
    const float t = expf(__fsub_rn(__fmul_rn(__ldg(row + c), 1.0e6f), m));
    s = __fadd_rn(s, t);
    if (c == cls) e = t;
  }
  return __fdiv_rn(e, s);
}

// hot value of class `cls` from a staged row.  Fast path: when the runner-up is more than 110 below the
// maximum (in units of 1e6 * logit) every other exp() is exactly 0 in float32, the sum is exactly 1 and the
// softmax is exactly one-hot — true for all but near-tie pixels.
__device__ __forceinline__ float hot_of_row(const float* row, int nc, int cls) {
  float m = -3.4e38f, m2 = -3.4e38f;
  int arg = 0;
  for (int c = 0; c < nc; ++c) {
    const float z = __fmul_rn(row[c], 1.0e6f);
    if (z > m) {
      m2 = m;
      m = z;
      arg = c;
    } else if (z > m2) {
      m2 = z;
    }
  }
  if (m - m2 > 110.f) return arg == cls ? 1.0f : 0.0f;
  float sum = 0.f, e = 0.f;
  for (int c = 0; c < nc; ++c) {
    const float t = expf(__fsub_rn(__fmul_rn(row[c], 1.0e6f), m));
    sum = __fadd_rn(sum, t);
    if (c == cls) e = t;
  }
  return __fdiv_rn(e, sum);
}

// same tiling and outputs as k_mask_bits (compaction.cuh), fed by the segmentation logits: the tile's
// [1024 x nc] floats are staged in shared memory with coalesced loads, then every thread classifies 4 pixels
// NC: classes when known at compile time (9: fully unrolled rows, all loads of the tile in flight), 0 = runtime.
// flag_onehot (forward call): cls9 bit 7 marks pixels whose softmax is exactly one-hot, so that the reduction need not
// read their logits again.
extern __shared__ __align__(16) float ls_smem[];
template <int NC>
__global__ void __launch_bounds__(256) k_ls_classify(const float* __restrict__ seg, WS ws, Dims d, LsWS lw, LsDims ld, int flag_onehot) {
  const int img = blockIdx.y, tile = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31;
  const int nc = NC ? NC : ld.nc;
  __shared__ int scnt[32];
  if (tid < 32) scnt[tid] = 0;
  const int p0 = tile * kCountTile;
  const int npx = min(kCountTile, d.hw - p0);
  const float* slab = seg + ((size_t)img * d.hw + p0) * nc;
  const int nfl = npx * nc;
  if (((nfl | (int)(((size_t)img * d.hw + p0) * nc)) & 3) == 0 && (reinterpret_cast<uintptr_t>(seg) & 15) == 0) {
    const float4* slab4 = reinterpret_cast<const float4*>(slab);  // 16-byte aligned slab: 128-bit loads
    float4* sm4 = reinterpret_cast<float4*>(ls_smem);
    if (NC && npx == kCountTile) {  // NC float4 per thread, all in flight before the first store
      float4 v[NC ? NC : 1];
#pragma unroll
      for (int u = 0; u < NC; ++u) v[u] = __ldg(slab4 + u * 256 + tid);
#pragma unroll
      for (int u = 0; u < NC; ++u) sm4[u * 256 + tid] = v[u];
    } else {
      for (int i = tid; i < nfl / 4; i += 256) sm4[i] = __ldg(slab4 + i);
    }
  } else {
    for (int i = tid; i < nfl; i += 256) ls_smem[i] = __ldg(slab + i);
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int q = k * 256 + tid;
    uint32_t m = 0;
    if (q < npx) {
      const float* row = ls_smem + q * nc;
      float mx = -3.4e38f, m2 = -3.4e38f;
      int arg = 0;
#pragma unroll
      for (int c = 0; c < nc; ++c) {
        const float z = __fmul_rn(row[c], 1.0e6f);
        if (z > mx) {
          m2 = mx;
          mx = z;
          arg = c;
        } else if (z > m2) {
          m2 = z;
        }
      }
      int c9 = 0;
      if (mx - m2 > 110.f) {  // exactly one-hot
        if (arg > 0) {
          m = 1u << (arg - 1);
          c9 = arg | (flag_onehot ? kOneHotFlag : 0);
        }
      } else {
        float sum = 0.f;
        for (int c = 0; c < nc; ++c) sum = __fadd_rn(sum, expf(__fsub_rn(__fmul_rn(row[c], 1.0e6f), mx)));
        for (int c = 1; c < nc; ++c) {
          const float hv = __fdiv_rn(expf(__fsub_rn(__fmul_rn(row[c], 1.0e6f), mx)), sum);
          m |= (uint32_t)(hv != 0.f) << (c - 1);
          if ((int)__fadd_rn(hv, 0.1f) == 1) c9 = c;  // :44 (at most one class can reach 0.9)
        }
      }
      ws.bits[(size_t)img * d.hw + p0 + q] = m;
      lw.cls9[(size_t)img * d.hw + p0 + q] = (unsigned char)c9;
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

// ---------------------------------------------------------------------------------- connected components
__device__ __forceinline__ int uf_find(int* parent, int x) {
  int r = x;
  while (true) {
    const int p = parent[r];
    if (p == r) break;
    r = p;
  }
  // path compression (racy but monotone: parent[i] <= i always and parents only ever decrease, so the walk
  // strictly descends and must stop at or below r even if other threads re-rooted the chain meanwhile)
  while (x > r) {
    const int p = parent[x];
    if (p > r) parent[x] = r;
    x = p;
  }
  return r;
}

__device__ __forceinline__ void uf_union(int* parent, int a, int b) {
  for (;;) {
    a = uf_find(parent, a);
    b = uf_find(parent, b);
    if (a == b) return;
    if (a < b) {
      const int t = a;
      a = b;
      b = t;
    }
    const int old = atomicMin(&parent[a], b);  // hang the larger root under the smaller one
    if (old == a) return;
    a = old;
  }
}

// The three union-find passes walk the compacted pixel lists of the jobs (grid (gx, J), raster order inside a
// list) instead of the whole image: only ~13 % of the pixels belong to any class.  A listed pixel is foreground
// of its job's class c iff cls9 == c + 1 (every such pixel is listed: int(hot + 0.1) == 1 implies hot != 0).
//
// k_cc_init: every foreground pixel starts under the first pixel of its horizontal run inside its warp's 32 list
// entries (runs are pre-merged with ballots, no atomics); its count is reset.
__global__ void __launch_bounds__(256) k_cc_init(WS ws, Dims d, LsWS lw, LsDims ld) {
  const int job = blockIdx.y, img = job / d.oc, c = job - img * d.oc;
  const int lane = threadIdx.x & 31;
  if (c == 0 && blockIdx.x == 0 && threadIdx.x == 0) lw.nroots[img] = 0;
  const int tn = ws.job_tn[job];
  const uint32_t* pix = ws.pix + (size_t)img * d.cap + ws.job_off[job];
  const unsigned char* cls = lw.cls9 + (size_t)img * ld.hw;
  for (int t0 = (blockIdx.x * 256 + threadIdx.x) & ~31; t0 < tn; t0 += gridDim.x * 256) {
    const int t = t0 + lane;
    uint32_t pk = 0xFFFFFFFFu;
    int p = -1;
    bool fg = false;
    if (t < tn) {
      pk = pix[t];
      p = (int)(pk >> 16) * ld.w + (int)(pk & 0xFFFFu);
      fg = cls[p] == c + 1;
    }
    const uint32_t pkl = __shfl_up_sync(0xffffffffu, pk, 1);
    const bool fgl = __shfl_up_sync(0xffffffffu, fg ? 1 : 0, 1) != 0;
    // the previous list entry is the left neighbour iff same row and x - 1 (packed values differ by one, x > 0)
    const bool joined = lane > 0 && fg && fgl && (pk & 0xFFFFu) != 0u && pkl + 1u == pk;
    const unsigned sb = __ballot_sync(0xffffffffu, !joined);
    const int sl = 31 - __clz(sb & (0xffffffffu >> (31 - lane)));  // nearest run start at or below this lane
    const int pstart = __shfl_sync(0xffffffffu, p, sl);
    if (fg) {
      lw.parent[(size_t)img * ld.hw + p] = pstart;
      lw.count[(size_t)img * ld.hw + p] = 0;
    }
  }
}

// Unions only where they are not implied: at the first entry of a warp's 32 list entries, and at the FIRST pixel
// of every horizontal overlap with the row above (left and upper-left neighbours both of the class => implied).
__global__ void __launch_bounds__(256) k_cc_merge(WS ws, Dims d, LsWS lw, LsDims ld) {
  const int job = blockIdx.y, img = job / d.oc, c = job - img * d.oc;
  const int lane = threadIdx.x & 31;
  const int tn = ws.job_tn[job];
  const uint32_t* pix = ws.pix + (size_t)img * d.cap + ws.job_off[job];
  const unsigned char* cls = lw.cls9 + (size_t)img * ld.hw;
  int* parent = lw.parent + (size_t)img * ld.hw;
  for (int t = blockIdx.x * 256 + threadIdx.x; t < tn; t += gridDim.x * 256) {
    const uint32_t pk = pix[t];
    const int x = pk & 0xFFFFu, y = pk >> 16, p = y * ld.w + x;
    if (cls[p] != c + 1) continue;
    const bool left = x > 0 && cls[p - 1] == c + 1;
    if (left && lane == 0) uf_union(parent, p, p - 1);  // k_cc_init joined runs inside the 32 entries only
    if (y > 0 && cls[p - ld.w] == c + 1) {
      const bool upleft = x > 0 && cls[p - ld.w - 1] == c + 1;
      if (!(left && upleft)) uf_union(parent, p, p - ld.w);
    }
  }
}

__global__ void __launch_bounds__(256) k_cc_flatten(WS ws, Dims d, LsWS lw, LsDims ld) {
  const int job = blockIdx.y, img = job / d.oc, c = job - img * d.oc;
  const int lane = threadIdx.x & 31;
  const int tn = ws.job_tn[job];
  const uint32_t* pix = ws.pix + (size_t)img * d.cap + ws.job_off[job];
  const unsigned char* cls = lw.cls9 + (size_t)img * ld.hw;
  int* parent = lw.parent + (size_t)img * ld.hw;
  for (int t0 = (blockIdx.x * 256 + threadIdx.x) & ~31; t0 < tn; t0 += gridDim.x * 256) {
    const int t = t0 + lane;
    int r = -1;
    bool fg = false;
    if (t < tn) {
      const uint32_t pk = pix[t];
      const int p = (int)(pk >> 16) * ld.w + (int)(pk & 0xFFFFu);
      fg = cls[p] == c + 1;
      if (fg) {
        r = uf_find(parent, p);
        parent[p] = r;
        if (r == p) lw.roots[(size_t)img * ld.hw + atomicAdd(&lw.nroots[img], 1)] = p;
      }
    }
    // component sizes: one atomic per distinct root in the warp (neighbouring pixels share their root)
    const unsigned same = __match_any_sync(0xffffffffu, r);
    if (fg && lane == __ffs(same) - 1) atomicAdd(&lw.count[(size_t)img * ld.hw + r], __popc(same));
  }
}

// Block-level end of the selection (:64-76): merges the per-thread top-3 lists (shuffle tree inside each warp, then
// thread 0 over the warp results), adds label 0 (every pixel outside the class's int mask), and returns — in thread 0 —
// the selected label as a root pixel index, -2 for label 0, -1 for a padding label that matches no pixel.
template <int NWARPS>
__device__ __forceinline__ int cc_pick(unsigned long long (&top)[3], int npix, int ncomp, const LsDims& ld) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    unsigned long long other[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) other[k] = __shfl_down_sync(0xffffffffu, top[k], o);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      unsigned long long key = other[k];
#pragma unroll
      for (int j = 0; j < 3; ++j)
        if (key > top[j]) {
          const unsigned long long t = top[j];
          top[j] = key;
          key = t;
        }
    }
  }
  npix = __reduce_add_sync(0xffffffffu, npix);
  ncomp = __reduce_add_sync(0xffffffffu, ncomp);
  __shared__ unsigned long long stop[NWARPS * 3];
  __shared__ int snp[NWARPS], snc[NWARPS];
  if (lane == 0) {
    for (int k = 0; k < 3; ++k) stop[warp * 3 + k] = top[k];
    snp[warp] = npix;
    snc[warp] = ncomp;
  }
  __syncthreads();
  int sel = -1;                         // padding label: matches no pixel
  if (tid == 0) {
    unsigned long long best[3] = {0ull, 0ull, 0ull};
    int tp = 0, tc = 0;
    for (int i = 0; i < NWARPS; ++i) {
      tp += snp[i];
      tc += snc[i];
      for (int k = 0; k < 3; ++k) {
        unsigned long long key = stop[i * 3 + k];
        if (key == 0ull) continue;
        for (int j = 0; j < 3; ++j)
          if (key > best[j]) {
            const unsigned long long t = best[j];
            best[j] = key;
            key = t;
          }
      }
    }
    const int bg = ld.hw - tp;  // label 0 of this class's int image
    const unsigned vbg = bg < ld.min_component ? 0u : (unsigned)bg;
    unsigned long long key = ((unsigned long long)vbg << 32) | 0xFFFFFFFFull;  // label 0: wins every tie
    for (int j = 0; j < 3; ++j)
      if (key > best[j]) {
        const unsigned long long t = best[j];
        best[j] = key;
        key = t;
      }
    if (ld.which < tc + 1) {            // real entries: label 0 and tc components
      const unsigned long long k = best[ld.which];
      const unsigned lab = 0xFFFFFFFFu - (unsigned)(k & 0xFFFFFFFFull);
      sel = lab == 0u ? -2 : (int)lab - 1;
    }
  }
  return sel;
}

// one block per (image, class): bincount -> threshold -> top_k -> pick index `which` (:64-76).
// Entries are label 0 (every pixel outside the class's int mask) and the components; the component with
// the smaller root pixel has the smaller tfa label.  key = (value << 32) | ~label : descending order.
__global__ void __launch_bounds__(256) k_cc_select(LsWS lw, LsDims ld) {
  const int job = blockIdx.x, img = job / ld.oc, c = job - img * ld.oc;
  const int tid = threadIdx.x;
  const int n = lw.nroots[img];
  const int* roots = lw.roots + (size_t)img * ld.hw;
  unsigned long long top[3] = {0ull, 0ull, 0ull};
  int npix = 0, ncomp = 0;
  for (int i = tid; i < n; i += 256) {
    const int r = roots[i];
    if (lw.cls9[(size_t)img * ld.hw + r] != c + 1) continue;
    const int cnt = lw.count[(size_t)img * ld.hw + r];
    npix += cnt;
    ++ncomp;
    const unsigned v = cnt < ld.min_component ? 0u : (unsigned)cnt;  // :66
    unsigned long long key = ((unsigned long long)v << 32) | (unsigned)(0xFFFFFFFFu - (unsigned)(r + 1));
    for (int k = 0; k < 3; ++k)
      if (key > top[k]) {
        const unsigned long long t = top[k];
        top[k] = key;
        key = t;
      }
  }
  const int sel = cc_pick<8>(top, npix, ncomp, ld);
  if (tid == 0) lw.sel[job] = sel;
}

// ---------------------------------------------------------------------------------- run-based components (forward)
// The forward call replaces k_cc_init / merge / flatten / select (63 us per 16 frames, global-memory union-find over
// pixels) by ONE kernel over horizontal runs: a job's raster-ordered pixel list is a sequence of runs (some hundred per
// object), the 4-connected components of the pixels are the components of the run-adjacency graph (runs of adjacent
// rows whose x ranges intersect), and a union-find over runs fits shared memory.  One block per job:
//   1. scan the list: run index of every entry (block-wide prefix of the run starts), run table (y, x0, x1);
//   2. every run looks up the runs of the row above that overlap it (binary search in the sorted table) and unions;
//   3. roots (smallest run = smallest pixel index = TFA's label order), component sizes;
//   4. the reference's selection (cc_pick);  5. the component mask of every list entry.
// Jobs with more than kCcRuns runs use the same code on run tables in global memory.
constexpr int kCcThreads = 512;
constexpr int kCcRuns = 2048;
constexpr int kCcPer = 4;  // list entries per thread and trip

__global__ void __launch_bounds__(kCcThreads) k_cc_runs(WS ws, Dims d, LsWS lw, LsDims ld) {
  const int job = blockIdx.x, img = job / d.oc, c = job - img * d.oc;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tn = ws.job_tn[job];
  const size_t lbase = (size_t)img * d.cap + ws.job_off[job];
  const uint32_t* pix = ws.pix + lbase;
  const unsigned char* cls = lw.cls9 + (size_t)img * ld.hw;
  int* ridx = lw.ridx + lbase;
  unsigned char* keep = lw.keep + lbase;
  __shared__ uint32_t s_pk[kCcRuns];
  __shared__ int s_x1[kCcRuns], s_parent[kCcRuns], s_cnt[kCcRuns];
  __shared__ int s_warp[kCcThreads / 32];
  __shared__ int s_sel;
  uint32_t* r_pk = s_pk;
  int *r_x1 = s_x1, *r_parent = s_parent, *r_cnt = s_cnt;
  int cap_runs = kCcRuns, nruns = 0;
  const unsigned char want = (unsigned char)(c + 1);
  for (int attempt = 0; attempt < 2; ++attempt) {
    int run0 = 0;  // runs that start in front of this trip (block-uniform)
    for (int base = 0; base < tn; base += kCcThreads * kCcPer) {
      // thread-contiguous entries t0 .. t0 + kCcPer - 1, plus the neighbours on either side
      const int t0 = base + tid * kCcPer;
      uint32_t pk[kCcPer + 2];
      bool fg[kCcPer + 2];
#pragma unroll
      for (int k = 0; k < kCcPer + 2; ++k) {
        const int t = t0 + k - 1;
        pk[k] = (t >= 0 && t < tn) ? __ldg(pix + t) : 0xFFFFFFFFu;
      }
#pragma unroll
      for (int k = 0; k < kCcPer + 2; ++k) {
        const int t = t0 + k - 1;
        fg[k] = (t >= 0 && t < tn) && (cls[(size_t)(pk[k] >> 16) * ld.w + (pk[k] & 0xFFFFu)] & kClassMask) == want;
      }
      int nstart = 0;
      bool start[kCcPer], last[kCcPer];
#pragma unroll
      for (int k = 1; k <= kCcPer; ++k) {
        // the previous list entry is the left neighbour iff same row and x - 1 (packed values differ by one, x > 0)
        const bool joined = fg[k] && fg[k - 1] && (pk[k] & 0xFFFFu) != 0u && pk[k - 1] + 1u == pk[k];
        const bool joined_next = fg[k] && fg[k + 1] && (pk[k + 1] & 0xFFFFu) != 0u && pk[k] + 1u == pk[k + 1];
        start[k - 1] = fg[k] && !joined;
        last[k - 1] = fg[k] && !joined_next;
        nstart += start[k - 1] ? 1 : 0;
      }
      int x = nstart;  // inclusive prefix of the run starts over the block
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
      }
      if (lane == 31) s_warp[warp] = x;
      __syncthreads();
      int woff = 0, total = 0;
#pragma unroll
      for (int k = 0; k < kCcThreads / 32; ++k) {
        const int v = s_warp[k];
        woff += k < warp ? v : 0;
        total += v;
      }
      int r = run0 + woff + x - nstart - 1;  // run of the entry in front of t0 (if it is foreground)
#pragma unroll
      for (int k = 0; k < kCcPer; ++k) {
        const int t = t0 + k;
        if (start[k]) {
          ++r;
          if (r < cap_runs) {
            r_pk[r] = pk[k + 1];
            r_parent[r] = r;
            r_cnt[r] = 0;
          }
        }
        if (last[k] && r < cap_runs) r_x1[r] = (int)(pk[k + 1] & 0xFFFFu);
        if (t < tn) ridx[t] = fg[k + 1] ? r : -1;
      }
      run0 += total;
      __syncthreads();  // s_warp is reused by the next trip
    }
    nruns = run0;
    if (nruns <= cap_runs) break;
    r_pk = lw.run_pk + lbase;  // more runs than shared memory holds: the same tables in global memory
    r_x1 = lw.run_x1 + lbase;
    r_parent = lw.run_parent + lbase;
    r_cnt = lw.run_cnt + lbase;
    cap_runs = 0x7fffffff;
    __syncthreads();
  }
  __syncthreads();
  // 2. unions with the overlapping runs of the row above
  for (int r = tid; r < nruns; r += kCcThreads) {
    const uint32_t pk = r_pk[r];
    const int y = pk >> 16, x0 = pk & 0xFFFFu, x1 = r_x1[r];
    if (y == 0) continue;
    const uint32_t key = ((uint32_t)(y - 1) << 16) | (uint32_t)x0;
    int lo = 0, hi = r;  // first run (in front of r) that starts at or behind (y - 1, x0)
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (r_pk[mid] < key) lo = mid + 1; else hi = mid;
    }
    int j = lo;
    if (j > 0 && (int)(r_pk[j - 1] >> 16) == y - 1) --j;  // the run that starts left of x0 may reach it
    for (; j < r; ++j) {
      const uint32_t pj = r_pk[j];
      if ((int)(pj >> 16) != y - 1 || (int)(pj & 0xFFFFu) > x1) break;
      if (r_x1[j] >= x0) uf_union(r_parent, r, j);
    }
  }
  __syncthreads();
  // 3. roots and component sizes
  for (int r = tid; r < nruns; r += kCcThreads) {
    const int root = uf_find(r_parent, r);
    atomicAdd(&r_cnt[root], r_x1[r] - (int)(r_pk[r] & 0xFFFFu) + 1);
  }
  __syncthreads();
  // 4. selection: entries are label 0 and the components; the component with the smaller root pixel has the smaller label
  unsigned long long top[3] = {0ull, 0ull, 0ull};
  int npix = 0, ncomp = 0;
  for (int r = tid; r < nruns; r += kCcThreads) {
    if (r_parent[r] != r) continue;
    const int cnt = r_cnt[r];
    npix += cnt;
    ++ncomp;
    const uint32_t pk = r_pk[r];
    const int rp = (int)(pk >> 16) * ld.w + (int)(pk & 0xFFFFu);
    const unsigned v = cnt < ld.min_component ? 0u : (unsigned)cnt;  // :66
    unsigned long long key = ((unsigned long long)v << 32) | (unsigned)(0xFFFFFFFFu - (unsigned)(rp + 1));
    for (int k = 0; k < 3; ++k)
      if (key > top[k]) {
        const unsigned long long t = top[k];
        top[k] = key;
        key = t;
      }
  }
  const int picked = cc_pick<kCcThreads / 32>(top, npix, ncomp, ld);
  if (tid == 0) {
    s_sel = picked;
    lw.sel[job] = picked;
  }
  __syncthreads();
  const int sel = s_sel;
  // 5. component mask of every list entry (copy_components, :72-79)
  for (int t = tid; t < tn; t += kCcThreads) {
    const int r = ridx[t];
    bool k = false;
    if (sel == -2) {
      k = r < 0;
    } else if (sel >= 0 && r >= 0) {
      const uint32_t pk = r_pk[uf_find(r_parent, r)];
      k = (int)(pk >> 16) * ld.w + (int)(pk & 0xFFFFu) == sel;
    }
    keep[t] = k ? 1 : 0;
  }
}

// ---------------------------------------------------------------------------------- weighted reduction
__device__ __forceinline__ float ls_weight(float x, int sigmoid_weights) {
  if (sigmoid_weights) return __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-x)));  // :33 (sigmoid_scale = 1)
  const float thr = 13.942385f;  // -(log(eps_f32) + 2), Eigen's softplus functor (:35)
  const float ex = expf(x);
  return x > thr ? x : (x < -thr ? ex : logf(__fadd_rn(ex, 1.0f)));
}

// One thread per listed pixel of a job: weight = hot_seg * component mask (:39-41, :72-79), and the pixel's
// confidence row turned into softplus / sigmoid weights (:32-35), stored keypoint-major like the directions.
__global__ void __launch_bounds__(256) k_ls_weights(WS ws, Dims d, LsWS lw, LsDims ld, const float* __restrict__ seg,
                                                    const float* __restrict__ conf) {
  const int job = blockIdx.y, img = job / d.oc, c = job - img * d.oc;
  const int tn = ws.job_tn[job];
  if (tn <= 0) return;
  const int off = ws.job_off[job];
  const uint32_t* pix = ws.pix + (size_t)img * d.cap + off;
  const int sel = ld.filter ? lw.sel[job] : 0;
  float* wt = lw.wt + (size_t)img * d.cap + off;
  float* cc = lw.cconf + ((size_t)img * d.cap + off) * d.vn;
  for (int t = blockIdx.x * 256 + threadIdx.x; t < tn; t += gridDim.x * 256) {
    const uint32_t pk = pix[t];
    const int x = pk & 0xFFFFu, y = pk >> 16;
    const size_t p = (size_t)img * ld.hw + (size_t)y * ld.w + x;
    float row[33];
    for (int k = 0; k < ld.nc; ++k) row[k] = __ldg(seg + p * ld.nc + k);
    float w = hot_of_row(row, ld.nc, c + 1);  // hot_seg (:39-41)
    if (ld.filter) {                          // copy_components * hot_seg (:72-79)
      const int c9 = lw.cls9[p];
      const bool keep = sel == -2 ? (c9 != c + 1) : (sel >= 0 && c9 == c + 1 && lw.parent[p] == sel);
      w = __fmul_rn(keep ? 1.0f : 0.0f, w);
    }
    wt[t] = w;
    // dropped pixels (weight 0) get defined zeros: k_ls_reduce loads the entry before it looks at the weight
    for (int v = 0; v < d.vn; ++v)
      cc[(size_t)v * tn + t] = w != 0.f ? ls_weight(__ldg(conf + p * ld.vn + v), ld.sigmoid_weights) : 0.f;
  }
}

// persistent over the refinement tiles: blockIdx.x strides over tiles, blockIdx.y = keypoint.  All operands
// come from the compact per-job arrays (pix, wt, vdir, cconf): coalesced, each read once.
__global__ void __launch_bounds__(256) k_ls_reduce(WS ws, Dims d, LsWS lw, LsDims ld) {
  const int v = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n_rtiles = ws.rtile_start[d.J];
  __shared__ double sred[8][5];
  const float fh = (float)ld.h;
  for (int rt = blockIdx.x; rt < n_rtiles; rt += gridDim.x) {
    const int job = ws.rtile_job[rt], tile = rt - ws.rtile_start[job];
    const int tn = ws.job_tn[job];
    const int img = job / d.oc;
    const size_t base = (size_t)img * d.cap + ws.job_off[job];
    const uint32_t* pix = ws.pix + base;
    const float* wt = lw.wt + base;
    const float2* vd = ws.vdir + base * d.vn + (size_t)v * tn;
    const float* cc = lw.cconf + base * d.vn + (size_t)v * tn;
    double s[5] = {0, 0, 0, 0, 0};
    // phase 1: all loads of the thread's 4 pixels in flight together; phase 2: arithmetic
    float lw_[kRefineTile / 256], lc_[kRefineTile / 256];
    uint32_t lp_[kRefineTile / 256];
    float2 ld_[kRefineTile / 256];
#pragma unroll
    for (int k = 0; k < kRefineTile / 256; ++k) {
      const int t = tile * kRefineTile + k * 256 + tid;
      const bool in = t < tn;
      lw_[k] = in ? wt[t] : 0.f;
      lp_[k] = in ? pix[t] : 0u;
      ld_[k] = in ? __ldg(vd + t) : make_float2(0.f, 0.f);  // (n0, n1) = (dy, dx)
      lc_[k] = in ? cc[t] : 0.f;  // (entries with weight 0 hold 0 and are skipped below)
    }
#pragma unroll
    for (int k = 0; k < kRefineTile / 256; ++k) {
      const float w = lw_[k];
      if (w == 0.f) continue;  // multiply_no_nan (:107-108); also positions past the end of the list
      const uint32_t pk = lp_[k];
      const int x = pk & 0xFFFFu, y = pk >> 16;
      const float2 dv = ld_[k];
      const float nrm = __fsqrt_rn(__fadd_rn(__fmul_rn(dv.x, dv.x), __fmul_rn(dv.y, dv.y)));  // :89
      const float n0 = nrm != 0.f ? __fdiv_rn(dv.x, nrm) : 0.f;  // divide_no_nan :90
      const float n1 = nrm != 0.f ? __fdiv_rn(dv.y, nrm) : 0.f;
      const float wc = lc_[k];
      const float r00 = __fmul_rn(__fsub_rn(1.0f, __fmul_rn(n0, n0)), wc);  // :92-94
      const float r01 = __fmul_rn(__fsub_rn(0.0f, __fmul_rn(n0, n1)), wc);
      const float r11 = __fmul_rn(__fsub_rn(1.0f, __fmul_rn(n1, n1)), wc);
      const float cy = __fdiv_rn(__fadd_rn((float)y, 0.5f), fh);  // :97  (both axes over the height)
      const float cx = __fdiv_rn(__fadd_rn((float)x, 0.5f), fh);  // :96
      const float q0 = __fadd_rn(__fmul_rn(r00, cy), __fmul_rn(r01, cx));  // :103-105
      const float q1 = __fadd_rn(__fmul_rn(r01, cy), __fmul_rn(r11, cx));
      s[0] += (double)__fmul_rn(r00, w);  // :108, :113
      s[1] += (double)__fmul_rn(r01, w);
      s[2] += (double)__fmul_rn(r11, w);
      s[3] += (double)__fmul_rn(q0, w);   // :107, :114
      s[4] += (double)__fmul_rn(q1, w);
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
      for (int k = 0; k < 8; ++k) t += sred[k][tid];
      ws.partial[((size_t)rt * d.vn + v) * 5 + tid] = t;
    }
    __syncthreads();
  }
}

// Forward pass without intermediates: weights, direction gather and the weighted reduction in ONE pass over the
// pixel lists.  blockIdx.x strides over the 1024-pixel tiles of the jobs, one warp per keypoint (block = 32 * vn).
//   phase 1 (all threads): weight = hot_seg * component mask of the tile's pixels (:39-41, :72-79) -> shared memory;
//   phase 2 (warp v):      keypoint v over the tile; the pixel's direction (8 bytes of its 72-byte row) and
//                          confidence logit are read straight from the dense network outputs — the rows of a tile
//                          are touched by all vn warps of the block back to back, so they cross HBM once — and
//                          go through the reference's float32 element-wise sequence (:89-108) into float64 sums.
// Replaces k_gather_dirs + k_ls_weights + k_ls_reduce (102 us of launches and 140 MB of intermediates per 16 frames)
// for the forward call; the backward pass still uses the gathered arrays.
// VEC (chosen on the host from the pointer): `direct` is 8-byte aligned and a pixel's (dy, dx) is one float2 load;
// otherwise (e.g. a view 4 bytes into an allocation) two scalar loads of the same floats.
constexpr int kFusedTile = 512;  // list entries per tile of k_ls_fused (d.rtile of the forward call)
template <bool VEC>
__global__ void __launch_bounds__(512, 2) k_ls_fused(WS ws, Dims d, LsWS lw, LsDims ld, const float* __restrict__ seg,
                                                  const float* __restrict__ direct, const float* __restrict__ conf,
                                                  int use_keep) {
  const int tid = threadIdx.x, lane = tid & 31, v = tid >> 5;
  const int n_rtiles = ws.rtile_start[d.J];
  __shared__ float s_w[kFusedTile];
  __shared__ uint32_t s_pix[kFusedTile];
  __shared__ float2 s_c[kFusedTile];  // grid position (cy, cx) = ((y+.5)/H, (x+.5)/H): one pair of divisions per pixel
  const float fh = (float)ld.h;
  for (int rt = blockIdx.x; rt < n_rtiles; rt += gridDim.x) {
    const int job = ws.rtile_job[rt], tile = rt - ws.rtile_start[job];
    const int tn = ws.job_tn[job];
    const int img = job / d.oc, c = job - img * d.oc;
    const size_t base = (size_t)img * d.cap + ws.job_off[job];
    const int sel = (ld.filter && !use_keep) ? lw.sel[job] : 0;
    const int npx = min(kFusedTile, tn - tile * kFusedTile);
    __syncthreads();  // the previous tile's readers are done with s_w / s_pix
    for (int k = tid; k < npx; k += blockDim.x) {
      const size_t le = base + (size_t)tile * kFusedTile + k;
      const uint32_t pk = ws.pix[le];
      const unsigned char kp = (ld.filter && use_keep) ? lw.keep[le] : (unsigned char)1;  // k_cc_runs' component mask
      const int x = pk & 0xFFFFu, y = pk >> 16;
      const size_t p = (size_t)img * ld.hw + (size_t)y * ld.w + x;
      const unsigned char c9raw = lw.cls9[p];
      const int c9 = c9raw & kClassMask;
      float w;
      if (c9raw & kOneHotFlag) {  // exactly one-hot softmax (k_ls_classify): hot_seg is 1 for the pixel's class, else 0
        w = c9 == c + 1 ? 1.0f : 0.0f;
      } else {
        float row[33];
        for (int q = 0; q < ld.nc; ++q) row[q] = __ldg(seg + p * ld.nc + q);
        w = hot_of_row(row, ld.nc, c + 1);  // hot_seg (:39-41)
      }
      if (ld.filter) {                          // copy_components * hot_seg (:72-79)
        const bool keep = use_keep ? kp != 0 : (sel == -2 ? (c9 != c + 1) : (sel >= 0 && c9 == c + 1 && lw.parent[p] == sel));
        w = __fmul_rn(keep ? 1.0f : 0.0f, w);
      }
      s_w[k] = w;
      s_pix[k] = pk;
      s_c[k] = make_float2(__fdiv_rn(__fadd_rn((float)y, 0.5f), fh), __fdiv_rn(__fadd_rn((float)x, 0.5f), fh));  // :96-97
    }
    __syncthreads();
    double s[5] = {0, 0, 0, 0, 0};
    constexpr int kBatch = 8;  // pixels per lane whose loads are in flight together (the loop is latency-bound otherwise)
    for (int k0 = 0; k0 < npx; k0 += 32 * kBatch) {
      float bw[kBatch], bc[kBatch];
      uint32_t bp[kBatch];
      float2 bd[kBatch];
#pragma unroll
      for (int j = 0; j < kBatch; ++j) {
        const int k = k0 + j * 32 + lane;
        bw[j] = k < npx ? s_w[k] : 0.f;
        bp[j] = k < npx ? s_pix[k] : 0u;
      }
#pragma unroll
      for (int j = 0; j < kBatch; ++j) {
        bd[j] = make_float2(0.f, 0.f);
        bc[j] = 0.f;
        if (bw[j] != 0.f) {
          const size_t p = (size_t)img * ld.hw + (size_t)(bp[j] >> 16) * ld.w + (bp[j] & 0xFFFFu);
          if (VEC) {
            bd[j] = __ldg(reinterpret_cast<const float2*>(direct + p * (size_t)(2 * d.vn)) + v);  // (n0, n1) = (dy, dx)
          } else {
            const float* dp = direct + p * (size_t)(2 * d.vn) + 2 * v;
            bd[j] = make_float2(__ldg(dp), __ldg(dp + 1));
          }
          bc[j] = __ldg(conf + p * (size_t)d.vn + v);
        }
      }
#pragma unroll
      for (int j = 0; j < kBatch; ++j) {
        const float w = bw[j];
        if (w == 0.f) continue;  // multiply_no_nan (:107-108); also slots past the end of the tile
        const float2 dv = bd[j];
        const float wc = ls_weight(bc[j], ld.sigmoid_weights);                                  // :32-35
        const float nrm = __fsqrt_rn(__fadd_rn(__fmul_rn(dv.x, dv.x), __fmul_rn(dv.y, dv.y)));  // :89
        const float n0 = nrm != 0.f ? __fdiv_rn(dv.x, nrm) : 0.f;  // divide_no_nan :90
        const float n1 = nrm != 0.f ? __fdiv_rn(dv.y, nrm) : 0.f;
        const float r00 = __fmul_rn(__fsub_rn(1.0f, __fmul_rn(n0, n0)), wc);  // :92-94
        const float r01 = __fmul_rn(__fsub_rn(0.0f, __fmul_rn(n0, n1)), wc);
        const float r11 = __fmul_rn(__fsub_rn(1.0f, __fmul_rn(n1, n1)), wc);
        const float2 g = s_c[k0 + j * 32 + lane];  // (w != 0 implies the slot is inside the tile)
        const float cy = g.x, cx = g.y;            // both axes over the height (:96-97)
        const float q0 = __fadd_rn(__fmul_rn(r00, cy), __fmul_rn(r01, cx));  // :103-105
        const float q1 = __fadd_rn(__fmul_rn(r01, cy), __fmul_rn(r11, cx));
        s[0] += (double)__fmul_rn(r00, w);  // :108, :113
        s[1] += (double)__fmul_rn(r01, w);
        s[2] += (double)__fmul_rn(r11, w);
        s[3] += (double)__fmul_rn(q0, w);   // :107, :114
        s[4] += (double)__fmul_rn(q1, w);
      }
    }
#pragma unroll
    for (int k = 0; k < 5; ++k) {
#pragma unroll
      for (int o = 16; o; o >>= 1) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
    }
    if (lane < 5) {
      double t = s[0];  // every lane holds all five sums after the xor tree
      t = lane == 1 ? s[1] : t;
      t = lane == 2 ? s[2] : t;
      t = lane == 3 ? s[3] : t;
      t = lane == 4 ? s[4] : t;
      ws.partial[((size_t)rt * d.vn + v) * 5 + lane] = t;
    }
  }
}

// Moore-Penrose inverse of the symmetric [[a,b],[b,c]] applied to (g0,g1); singular values below
// rcond * max are dropped (tf.linalg.pinv default rcond = 10 * 2 * eps_f64, :116)
__device__ __forceinline__ void pinv2x2_apply(double a, double b, double c, double g0, double g1, double& p0, double& p1) {
  const double m = 0.5 * (a + c), dd = 0.5 * (a - c);
  const double r = sqrt(dd * dd + b * b);
  const double l1 = m + r, l2 = m - r;  // eigenvalues, l1 >= l2
  const double smax = fmax(fabs(l1), fabs(l2));
  const double cut = 4.440892098500626e-15 * smax;
  p0 = p1 = 0.0;
  if (!(smax > 0.0)) {
    if (smax != smax) p0 = p1 = smax;  // NaN in, NaN out
    return;
  }
  if (fabs(l1) > cut && fabs(l2) > cut) {
    const double det = a * c - b * b;
    p0 = (c * g0 - b * g1) / det;
    p1 = (a * g1 - b * g0) / det;
    return;
  }
  // rank one: project on the eigenvector of the dominant eigenvalue
  const double l = fabs(l1) >= fabs(l2) ? l1 : l2;
  double vx = b, vy = l - a;
  if (fabs(l - c) > fabs(vy)) {
    vx = l - c;
    vy = b;
  }
  const double nn = vx * vx + vy * vy;
  if (!(nn > 0.0)) {  // diagonal matrix with one zero entry
    if (fabs(a) >= fabs(c)) p0 = g0 / a; else p1 = g1 / c;
    return;
  }
  const double proj = (vx * g0 + vy * g1) / (nn * l);
  p0 = vx * proj;
  p1 = vy * proj;
}

// one warp per job, lane v = keypoint
__global__ void __launch_bounds__(32) k_ls_solve(WS ws, Dims d, LsDims ld, float* __restrict__ out, double* dbg_sums, uint32_t* sticky) {
  const int job = blockIdx.x, v = threadIdx.x;
  if (job == 0 && v == 0 && sticky) {  // a pixel-list overflow (raised by k_place) must not stay silent: -> casa_sync
    const unsigned st = (unsigned)ws.ctrl[CTRL_STATUS] & CASA_STATUS_PIX_OVERFLOW;
    if (st) atomicOr(sticky, st);
  }
  if (v >= d.vn) return;
  const int r0 = ws.rtile_start[job], r1 = ws.rtile_start[job + 1];
  double acc[5] = {0, 0, 0, 0, 0};
  for (int rt = r0; rt < r1; ++rt)
#pragma unroll
    for (int k = 0; k < 5; ++k) acc[k] += ws.partial[((size_t)rt * d.vn + v) * 5 + k];
  double p0, p1;
  pinv2x2_apply(acc[0], acc[1], acc[2], acc[3], acc[4], p0, p1);
  const float o0 = __fmul_rn((float)p0, (float)ld.h), o1 = __fmul_rn((float)p1, (float)ld.h);  // :122
  bool bad = false;
#pragma unroll
  for (int k = 0; k < 5; ++k) bad |= !(fabs(acc[k]) <= 1.7e308);
  bad |= !(fabsf(o0) <= 3.4e38f) || !(fabsf(o1) <= 3.4e38f);
  if (bad) {
    atomicOr(reinterpret_cast<unsigned*>(&ws.ctrl[CTRL_STATUS]), LS_STATUS_NONFINITE);
    if (sticky) atomicOr(sticky, LS_STATUS_NONFINITE);
  }
  out[((size_t)job * d.vn + v) * 2] = o0;  // (y, x) pixels; scalar stores: out need only be 4-byte aligned
  out[((size_t)job * d.vn + v) * 2 + 1] = o1;
  if (dbg_sums)
#pragma unroll
    for (int k = 0; k < 5; ++k) dbg_sums[((size_t)job * d.vn + v) * 5 + k] = acc[k];
}

// ---------------------------------------------------------------------------------------------- backward
// Gradient of the layer output w.r.t. `direct` and the confidence logits (SURVEY.md section 8f-4; the layer is
// differentiated at /root/reference/train_casapose.py:536-595, seg is behind tf.stop_gradient :37).
//
// k_ls_adjoint: per (job, keypoint), float64.  With A = sum hot*R, b = sum hot*q, P = pinv(A), x = P b and the
// incoming g = dL/dp = grad_out * height (:122):   dL/db = P g =: lam;   dL/dA = -lam x^T + v u^T + r s^T with
// u = P lam, v = (I - A P) b, r = P x, s = (I - A P) g  (differential of the pseudo-inverse at constant rank; the
// last two terms vanish when A is invertible).  Stored as float32 — the gradient passes back through the
// float32 -> float64 casts of :113-114.
__global__ void __launch_bounds__(32) k_ls_adjoint(WS ws, Dims d, LsDims ld, const float* __restrict__ grad_out,
                                                   float* __restrict__ adj) {
  const int job = blockIdx.x, v = threadIdx.x;
  if (v >= d.vn) return;
  const int r0 = ws.rtile_start[job], r1 = ws.rtile_start[job + 1];
  double acc[5] = {0, 0, 0, 0, 0};
  for (int rt = r0; rt < r1; ++rt)
#pragma unroll
    for (int k = 0; k < 5; ++k) acc[k] += ws.partial[((size_t)rt * d.vn + v) * 5 + k];
  const double a = acc[0], b = acc[1], c = acc[2], q0 = acc[3], q1 = acc[4];
  double P00, P10, P01, P11;
  pinv2x2_apply(a, b, c, 1.0, 0.0, P00, P10);
  pinv2x2_apply(a, b, c, 0.0, 1.0, P01, P11);
  const float* go = grad_out + ((size_t)job * d.vn + v) * 2;  // scalar loads: grad_out need only be 4-byte aligned
  const double g0 = (double)__fmul_rn(go[0], (float)ld.h), g1 = (double)__fmul_rn(go[1], (float)ld.h);
  const double x0 = P00 * q0 + P01 * q1, x1 = P10 * q0 + P11 * q1;
  const double l0 = P00 * g0 + P10 * g1, l1 = P01 * g0 + P11 * g1;  // P^T g
  // I - A P (A symmetric)
  const double e00 = 1.0 - (a * P00 + b * P10), e01 = -(a * P01 + b * P11);
  const double e10 = -(b * P00 + c * P10), e11 = 1.0 - (b * P01 + c * P11);
  const double u0 = P00 * l0 + P01 * l1, u1 = P10 * l0 + P11 * l1;          // P P^T g
  const double v0 = e00 * q0 + e01 * q1, v1 = e10 * q0 + e11 * q1;          // (I - A P) b
  const double rr0 = P00 * x0 + P10 * x1, rr1 = P01 * x0 + P11 * x1;        // P^T P b
  const double s0 = e00 * g0 + e10 * g1, s1 = e01 * g0 + e11 * g1;          // (I - P A)^T g = (I - A P)^T g ... transposed index
  float* o = adj + ((size_t)job * d.vn + v) * 6;
  o[0] = (float)(-l0 * x0 + v0 * u0 + rr0 * s0);
  o[1] = (float)(-l0 * x1 + v0 * u1 + rr0 * s1);
  o[2] = (float)(-l1 * x0 + v1 * u0 + rr1 * s0);
  o[3] = (float)(-l1 * x1 + v1 * u1 + rr1 * s1);
  o[4] = (float)l0;
  o[5] = (float)l1;
}

// blockIdx.x strides over the refinement tiles (all keypoints per thread: 72 + 36 contiguous bytes per pixel).
// grad_direct [b,h,w,2*vn] and grad_conf [b,h,w,vn] must be zero-filled; pixels listed for one class are
// stored, pixels listed for several (near-tie logits) are accumulated atomically.  VEC (chosen on the host): grad_direct
// is 8-byte aligned and a pixel's (dy, dx) gradient is one float2 store, otherwise two scalar stores.
template <bool VEC>
__global__ void __launch_bounds__(256) k_ls_backward(WS ws, Dims d, LsWS lw, LsDims ld, const float* __restrict__ adj,
                                                     float* __restrict__ grad_direct, float* __restrict__ grad_conf) {
  const int tid = threadIdx.x;
  const int n_rtiles = ws.rtile_start[d.J];
  __shared__ float sadj[32 * 6];
  const float fh = (float)ld.h;
  for (int rt = blockIdx.x; rt < n_rtiles; rt += gridDim.x) {
    const int job = ws.rtile_job[rt], tile = rt - ws.rtile_start[job];
    const int tn = ws.job_tn[job];
    const int img = job / d.oc;
    const size_t base = (size_t)img * d.cap + ws.job_off[job];
    __syncthreads();
    if (tid < d.vn * 6) sadj[tid] = adj[(size_t)job * d.vn * 6 + tid];
    __syncthreads();
#pragma unroll 1
    for (int k = 0; k < kRefineTile / 256; ++k) {
      const int t = tile * kRefineTile + k * 256 + tid;
      if (t >= tn) continue;
      const float hw = lw.wt[base + t];
      if (hw == 0.f) continue;  // multiply_no_nan: no gradient through pixels with hot == 0
      const uint32_t pk = ws.pix[base + t];
      const int x = pk & 0xFFFFu, y = pk >> 16;
      const size_t p = (size_t)img * ld.hw + (size_t)y * ld.w + x;
      const bool shared_px = __popc(ws.bits[p]) > 1;
      const float cy = __fdiv_rn(__fadd_rn((float)y, 0.5f), fh), cx = __fdiv_rn(__fadd_rn((float)x, 0.5f), fh);
      for (int v = 0; v < d.vn; ++v) {
        const float2 dv = __ldg(ws.vdir + base * d.vn + (size_t)v * tn + t);
        const float wc = lw.cconf[base * d.vn + (size_t)v * tn + t];
        const float nrm = __fsqrt_rn(__fadd_rn(__fmul_rn(dv.x, dv.x), __fmul_rn(dv.y, dv.y)));
        const float inv = nrm != 0.f ? __fdiv_rn(1.0f, nrm) : 0.f;
        const float n0 = dv.x * inv, n1 = dv.y * inv;
        const float* A = sadj + v * 6;
        // G = hot * (Abar + lam p^T): gradient w.r.t. R_full of this pixel (:103-108)
        const float G00 = hw * (A[0] + A[4] * cy), G01 = hw * (A[1] + A[4] * cx);
        const float G10 = hw * (A[2] + A[5] * cy), G11 = hw * (A[3] + A[5] * cx);
        const float M00 = 1.0f - n0 * n0, M01 = -n0 * n1, M11 = 1.0f - n1 * n1;
        const float gw = G00 * M00 + (G01 + G10) * M01 + G11 * M11;  // d/dw of R_full = M * w (:94)
        // M = I - n n^T (:92-93): dL/dn = -(G_M + G_M^T) n, G_M = w G
        const float gn0 = -wc * (2.0f * G00 * n0 + (G01 + G10) * n1);
        const float gn1 = -wc * ((G01 + G10) * n0 + 2.0f * G11 * n1);
        // n = d / |d| (:89-90): dL/dd = (gn - (gn . n) n) / |d|; zero vector -> zero gradient (divide_no_nan)
        const float dot = gn0 * n0 + gn1 * n1;
        const float gd0 = (gn0 - dot * n0) * inv, gd1 = (gn1 - dot * n1) * inv;
        // softplus' = sigmoid = 1 - exp(-softplus) (:35);  sigmoid' = s (1 - s) (:33)
        const float gc = gw * (ld.sigmoid_weights ? wc * (1.0f - wc) : -expm1f(-wc));
        float* gdp = grad_direct + p * (size_t)(2 * d.vn) + 2 * v;
        float* gcp = grad_conf + p * (size_t)d.vn + v;
        if (shared_px) {
          atomicAdd(gdp, gd0);
          atomicAdd(gdp + 1, gd1);
          atomicAdd(gcp, gc);
        } else {
          if (VEC) {
            *reinterpret_cast<float2*>(gdp) = make_float2(gd0, gd1);
          } else {
            gdp[0] = gd0;
            gdp[1] = gd1;
          }
          *gcp = gc;
        }
      }
    }
  }
}

}  // namespace casa
