// Target assignment for a batch of images: IoU matching with the reference's greedy forced
// assignment + threshold matching + offset encoding, one CTA per image (persistent grid).
//
// Reference semantics reproduced bit for bit (utils/bbox.py:44-101, models/ssd_model.py:211-224):
//   * IoU in the reference's exact operation order and dtype mix (iou_corners, common.cuh).
//   * Phase 1 (utils/bbox.py:62-68): T rounds of whole-matrix first-arg-max with row+column
//     knock-out (knocked-out entries read as 0.0 and still take part in the arg-max).
//   * Phase 2 (:71-79) == for every prior not taken in phase 1: first-arg-max ground truth over
//     ALL rows, positive iff not (iou <= thresh).
//   * Scatter (:84-90) in append order, later pairs overwrite; encode (:94-101).
//
// How the work is organised (32 priors = one tile; with a prior index every tile holds priors of one
// shape in a compact block, so the per-tile statistics give a tight bound):
//   search   one WARP per ground-truth row.  The warp bounds, for every tile, the IoU any of its priors
//            can reach (conservative float upper bound from the tile statistics), evaluates the tile
//            with the highest bound first, then every tile whose bound still reaches
//            min(thresh, running row maximum): only those can hold a positive or the row's arg-max.
//            Evaluation is the exact float64 formula, lane = prior.  The row maximum / first arg-max
//            column live in the warp's registers (no atomics, no log); pairs above the threshold are
//            appended to a small per-image list.
//   columns  the list is reduced to each prior's first-arg-max row (phase 2) with two rounds of
//            atomics on a per-CTA scratch that is only ever touched at listed priors.
//   greedy   warp 0 runs the T rounds on the cached row maxima (rows cached in registers); rows whose
//            cached column was just taken by another row are searched again over the live columns.
//   output   every prior is written once, coalesced in prior order: unmatched rows copy a precomputed
//            encoding (prior index) or compute it, positives encode their ground truth; the phase-1
//            pairs overwrite last.
#include <math_constants.h>
#include <algorithm>
#include <map>
#include <mutex>
#include <unordered_map>
#include <utility>
#include <vector>
#include "common.cuh"

namespace ssdg {

constexpr int kMatchThreads = 512;
constexpr int kMatchCtasPerSm = 2;
constexpr int kMatchMaxCtas = 1024;
constexpr int kCandCap = 8192;          // listed (row, prior) pairs above the threshold per image
constexpr int kABits = 21;
constexpr int kMaxGT = 2048;
constexpr int kTileSmemMax = 1024;      // tile statistics staged in shared memory up to this many tiles
constexpr int kSuper = 8;               // tiles per super-tile (two-level bound of the row search)
constexpr int kSuperRegs = kTileSmemMax / kSuper / 32;   // super-tile bounds a lane keeps in registers (4)
constexpr int kElimSmemWords = 4096;    // 16 KB: bitmaps in shared memory up to 131072 priors

struct TileStat {
  float x1, y1, x2, y2;   // bounding box of the tile's priors, rounded outwards
  float wmax, hmax;       // largest corner-derived width / height (rounded up)
  float amin;             // smallest area (rounded down)
  u32 safe;               // 1: every prior of the tile is finite
  float cx1, cy1, cx2, cy2;   // range of the priors' corner mid-points (rounded outwards)
};

struct Cand {
  u64 key;
  int a, t;
};

struct MatchParams {
  const void* gt_boxes;
  const float* gt_cls;
  const int* gt_off;
  const void* priors;
  int B, A, max_gt, tm;  // tm = max_gt rounded up to 32
  double thresh;
  int* out_cls;
  float* out_box;
  float* out_loc;
  uint8_t* out_mask;
  int* out_match;
  u32* ws_head;             // [0] next image, [1] status bits, [2] next row of the search kernel, [3] tiles evaluated
  u32* ws_ncand;            // [B] listed pairs of the image
  u64* ws_rowkey;           // [B*tm] row maximum (key64) found by the search kernel
  int* ws_rowcol;           // [B*tm] its first arg-max prior
  Cand* ws_cand;            // per image kCandCap
  u64* ws_colkey;           // per CTA A
  int* ws_colt;             // per CTA A
  u32* ws_bits;             // per CTA 2*elim_words (knocked-out columns, touched columns) when not in smem
  const TileStat* tiles;    // [ntiles]
  const TileStat* supers;   // [ceil(ntiles / kSuper)] statistics of kSuper consecutive tiles each
  const int* perm;          // [ntiles*32] slot -> prior index (-1: padding); NULL: identity
  const void* pprior;       // [ntiles*32,4] the priors in slot order (same dtype); NULL: gather through perm
  const float4* unmatched;  // [A] encoding of an all-zero box per prior; NULL: compute
  int ntiles;
  int elim_words;
  int bits_in_smem;
  u64 index_sum;            // content checksum of the priors the index was built from (0: no index)
  long long prior_words;    // 8-byte words of the prior array
};

// Position-weighted sum of the 8-byte words of the prior array (mod 2^64): order-independent to accumulate, sensitive
// to any changed, moved or swapped word.  Host (index build) and device (every launch with an index) agree exactly.
__host__ __device__ __forceinline__ u64 checksum_term(u64 word, long long i) { return word * (2ull * (u64)i + 1ull); }

template <typename TG, typename TP>
struct Promote {
  typedef double type;
};
template <>
struct Promote<float, float> {
  typedef float type;
};

template <typename T>
struct Vec4;
template <>
struct Vec4<float> {
  static __device__ __forceinline__ void load(const void* base, long long i, float& a, float& b, float& c,
                                              float& d) {
    float4 v = __ldg(reinterpret_cast<const float4*>(base) + i);
    a = v.x; b = v.y; c = v.z; d = v.w;
  }
};
template <>
struct Vec4<double> {
  static __device__ __forceinline__ void load(const void* base, long long i, double& a, double& b, double& c,
                                              double& d) {
    const double2* p = reinterpret_cast<const double2*>(base) + 2 * i;
    double2 u = __ldg(p), v = __ldg(p + 1);
    a = u.x; b = u.y; c = v.x; d = v.y;
  }
};

__device__ __forceinline__ float f_down(double v) { return __double2float_rd(v); }
__device__ __forceinline__ float f_up(double v) { return __double2float_ru(v); }
__device__ __forceinline__ bool finite4(double a, double b, double c, double d) {
  return isfinite(a) && isfinite(b) && isfinite(c) && isfinite(d);
}

// apply_anchor_box for one row (utils/bbox.py:98-99), float64 arithmetic, float32 result
// (the TensorSpec cast at models/ssd_model.py:222).
template <typename TP>
__device__ __forceinline__ float4 encode_row(float bx, float by, float bw, float bh, TP dx, TP dy, TP dw,
                                             TP dh) {
  double tx = ((double)bx - (double)dx) / (double)dw;
  double ty = ((double)by - (double)dy) / (double)dh;
  double rw = (double)fmaxf(bw, 1e-5f) / (double)max_nn(dw, (TP)1e-5);
  double rh = (double)fmaxf(bh, 1e-5f) / (double)max_nn(dh, (TP)1e-5);
  return make_float4((float)tx, (float)ty, (float)log(rw), (float)log(rh));
}

// Conservative float bound of the IoU the exact path would compute for a ground truth against any prior
// of a tile: iub bounds the intersection from above, dlb the denominator from below (outward-rounded
// corners, directed rounding).  A NaN anywhere leaves dlb NaN.
__device__ __forceinline__ void iou_bound(const float4& g, float ga_lo, const TileStat& s, float& iub, float& dlb) {
  float ex = fmaxf(__fsub_ru(fminf(g.z, s.x2), fmaxf(g.x, s.x1)), 1.0001e-10f);
  float ey = fmaxf(__fsub_ru(fminf(g.w, s.y2), fmaxf(g.y, s.y1)), 1.0001e-10f);
  // a prior with mid-point c and half-extent h overlaps the ground truth by at most  g.hi - (c - h)  and
  // (c + h) - g.lo:  bound both with the tile's mid-point range
  const float hw = s.wmax * 0.50001f, hh = s.hmax * 0.50001f;
  ex = fminf(ex, fminf(__fadd_ru(__fsub_ru(g.z, s.cx1), hw), __fsub_ru(__fadd_ru(s.cx2, hw), g.x)));
  ey = fminf(ey, fminf(__fadd_ru(__fsub_ru(g.w, s.cy1), hh), __fsub_ru(__fadd_ru(s.cy2, hh), g.y)));
  ex = fmaxf(fminf(ex, s.wmax), 1.0001e-10f);
  ey = fmaxf(fminf(ey, s.hmax), 1.0001e-10f);
  iub = __fmul_ru(ex, ey);
  dlb = __fadd_rd(__fsub_rd(__fadd_rd(ga_lo, s.amin), iub), 0.9999e-10f);
}
// true unless  iou < bound  is certain for every prior of the tile
__device__ __forceinline__ bool may_reach(const float4& g, float ga_lo, const TileStat& s, float bound) {
  float iub, dlb;
  iou_bound(g, ga_lo, s, iub, dlb);
  return !s.safe || !(dlb > 0.f && iub * 1.0001f < bound * dlb);
}

// ---- per-tile statistics of the priors ---------------------------------------------------------------------
template <typename TP>
__global__ void __launch_bounds__(256) tile_stats_kernel(const void* __restrict__ priors, int A, const int* __restrict__ perm,
                                                         int ntiles, TileStat* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int tile = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (tile >= ntiles) return;
  const int slot = (tile << 5) + lane;
  const int a = perm ? perm[slot] : slot;
  const bool valid = a >= 0 && a < A;
  u32 kx1 = ~0u, ky1 = ~0u, kx2 = 0u, ky2 = 0u, kw = 0u, kh = 0u, ka = ~0u;
  u32 kc1 = ~0u, kd1 = ~0u, kc2 = 0u, kd2 = 0u;
  bool safe = true;
  if (valid) {
    TP cx, cy, w, h;
    Vec4<TP>::load(priors, a, cx, cy, w, h);
    Corners<TP> c = corners_of<TP>(cx, cy, w, h);
    safe = finite4((double)c.x1, (double)c.y1, (double)c.x2, (double)c.y2) && isfinite((double)c.area);
    if (safe) {
      const float x1 = f_down((double)c.x1), y1 = f_down((double)c.y1);
      const float x2 = f_up((double)c.x2), y2 = f_up((double)c.y2);
      kx1 = key32(x1); ky1 = key32(y1); kx2 = key32(x2); ky2 = key32(y2);
      kw = key32(__fsub_ru(x2, x1)); kh = key32(__fsub_ru(y2, y1));
      ka = key32(f_down((double)c.area));
      const double mx = 0.5 * ((double)c.x1 + (double)c.x2), my = 0.5 * ((double)c.y1 + (double)c.y2);
      kc1 = key32(f_down(mx - 1e-12 * fabs(mx))); kc2 = key32(f_up(mx + 1e-12 * fabs(mx)));
      kd1 = key32(f_down(my - 1e-12 * fabs(my))); kd2 = key32(f_up(my + 1e-12 * fabs(my)));
    }
  }
  TileStat st;
  st.cx1 = unkey32(__reduce_min_sync(SSDG_FULL, kc1));
  st.cy1 = unkey32(__reduce_min_sync(SSDG_FULL, kd1));
  st.cx2 = unkey32(__reduce_max_sync(SSDG_FULL, kc2));
  st.cy2 = unkey32(__reduce_max_sync(SSDG_FULL, kd2));
  st.x1 = unkey32(__reduce_min_sync(SSDG_FULL, kx1));
  st.y1 = unkey32(__reduce_min_sync(SSDG_FULL, ky1));
  st.x2 = unkey32(__reduce_max_sync(SSDG_FULL, kx2));
  st.y2 = unkey32(__reduce_max_sync(SSDG_FULL, ky2));
  st.wmax = fmaxf(unkey32(__reduce_max_sync(SSDG_FULL, kw)), 1.0001e-10f);
  st.hmax = fmaxf(unkey32(__reduce_max_sync(SSDG_FULL, kh)), 1.0001e-10f);
  st.amin = unkey32(__reduce_min_sync(SSDG_FULL, ka));
  st.safe = __all_sync(SSDG_FULL, safe) ? 1u : 0u;
  if (lane == 0) out[tile] = st;
}

// statistics of kSuper consecutive tiles: every field moves the way that can only raise the tile bound
__global__ void __launch_bounds__(128) super_stats_kernel(const TileStat* __restrict__ tiles, int ntiles, TileStat* __restrict__ out) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s * kSuper >= ntiles) return;
  TileStat u = tiles[s * kSuper];
  for (int k = 1; k < kSuper && s * kSuper + k < ntiles; ++k) {
    const TileStat v = tiles[s * kSuper + k];
    u.x1 = fminf(u.x1, v.x1); u.y1 = fminf(u.y1, v.y1); u.x2 = fmaxf(u.x2, v.x2); u.y2 = fmaxf(u.y2, v.y2);
    u.wmax = fmaxf(u.wmax, v.wmax); u.hmax = fmaxf(u.hmax, v.hmax); u.amin = fminf(u.amin, v.amin);
    u.safe = u.safe & v.safe;
    u.cx1 = fminf(u.cx1, v.cx1); u.cy1 = fminf(u.cy1, v.cy1); u.cx2 = fmaxf(u.cx2, v.cx2); u.cy2 = fmaxf(u.cy2, v.cy2);
  }
  out[s] = u;
}

// encoding of an all-zero (unmatched) box against every prior (utils/bbox.py:85,98-99)
template <typename TP>
__global__ void __launch_bounds__(256) unmatched_kernel(const void* __restrict__ priors, int A, float4* __restrict__ out) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= A) return;
  TP dx, dy, dw, dh;
  Vec4<TP>::load(priors, a, dx, dy, dw, dh);
  out[a] = encode_row<TP>(0.f, 0.f, 0.f, 0.f, dx, dy, dw, dh);
}

template <typename TG, typename TP>
struct MatchSmem {
  typedef typename Promote<TG, TP>::type R;
  R *gx1, *gy1, *gx2, *gy2, *ga;     // ground-truth corners / area in the result dtype
  float4* cbox;                      // outward-rounded float box of the ground truth
  float* galo;                       // float lower bound of the area (NaN: never cull)
  u64* rowkey;                       // cached row maximum (key64) over live columns
  int* rowcol;                       // first arg-max column of rowkey
  int *pair_t, *pair_a, *rs_list, *order;
  uint8_t* dead;
  int* red_idx;
  int* ctl;                          // control words, see enum
  TileStat* tiles_s;                 // staged tile statistics (when they fit)
  u32 *elim_s, *touch_s;             // bitmaps (when they fit)
  __device__ void carve(unsigned char* base, int tm, int ntiles_s, int bit_words) {
    size_t o = 0;
    gx1 = (R*)(base + o); o += sizeof(R) * tm;
    gy1 = (R*)(base + o); o += sizeof(R) * tm;
    gx2 = (R*)(base + o); o += sizeof(R) * tm;
    gy2 = (R*)(base + o); o += sizeof(R) * tm;
    ga = (R*)(base + o); o += sizeof(R) * tm;
    o = (o + 15) & ~(size_t)15;
    cbox = (float4*)(base + o); o += 16 * (size_t)tm;
    tiles_s = (TileStat*)(base + o); o += sizeof(TileStat) * (size_t)ntiles_s;
    rowkey = (u64*)(base + o); o += 8 * (size_t)tm;
    galo = (float*)(base + o); o += 4 * (size_t)tm;
    rowcol = (int*)(base + o); o += 4 * (size_t)tm;
    pair_t = (int*)(base + o); o += 4 * (size_t)tm;
    pair_a = (int*)(base + o); o += 4 * (size_t)tm;
    rs_list = (int*)(base + o); o += 4 * (size_t)tm;
    order = (int*)(base + o); o += 4 * (size_t)tm;
    red_idx = (int*)(base + o); o += 4 * 4;
    ctl = (int*)(base + o); o += 4 * 16;
    elim_s = (u32*)(base + o); o += 4 * (size_t)bit_words;
    touch_s = (u32*)(base + o); o += 4 * (size_t)bit_words;
    dead = (uint8_t*)(base + o);
  }
};
static size_t match_smem_bytes(int tm, int ntiles_s, int bit_words) {
  return (size_t)tm * (5 * 8 + 16 + 8 + 4 + 20 + 1) + (size_t)ntiles_s * sizeof(TileStat) +
         (size_t)bit_words * 8 + 16 + 64 + 96;
}

// ---- search: the row maxima of the whole batch --------------------------------------------------------------
// One warp per ground-truth ROW, rows handed out dynamically over the whole batch (they differ in cost and the
// images in row count): small CTAs that fill every SM evenly and fit beside the streaming kernels of the other
// branch.  Per row: the first arg-max prior (exact formula) and every pair above the threshold, appended to the
// image's list.  The per-image kernel below consumes both.
constexpr int kSearchThreads = 128;
constexpr int kSearchWarps = kSearchThreads / 32;
// 10 CTAs per SM (48 registers): four instead of three of them fit beside a filter CTA of the other branch
// (chained step 0.513 -> 0.508 ms; alone 0.141 -> 0.139 ms).  Both the launch bounds and the grid use it.
constexpr int kSearchCtasPerSm = 10;

template <typename TG, typename TP, bool kHier>   // kHier: two-level bound (super-tiles of kSuper tiles, then tiles); up to kTileSmemMax tiles
__global__ void __launch_bounds__(kSearchThreads, kSearchCtasPerSm) search_kernel(MatchParams P) {
  typedef typename Promote<TG, TP>::type R;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31;
  const int A = P.A, ntiles = P.ntiles;
  // the tile statistics stay in global memory (L1/L2-resident, 14 KB for SSD300): staging them per CTA costs
  // shared memory that decides how many of these CTAs fit beside a streaming kernel of the other branch
  const TileStat* tiles = P.tiles;
  const R EPS = (R)1e-10;
  const u64 thr_key = key64((double)(R)P.thresh);
  const float thr_lo = f_down((double)(R)P.thresh);
  const int total_rows = P.gt_off[P.B];
  u32 n_eval = 0u;   // tiles this warp evaluated exactly (ws_head[3]: the matcher's work counter, bench.py)
  for (;;) {
    int gr = 0;
    if (lane == 0) gr = (int)atomicAdd(&P.ws_head[2], 1u);
    gr = __shfl_sync(SSDG_FULL, gr, 0);
    if (gr >= total_rows) {
      if (lane == 0 && n_eval) atomicAdd(&P.ws_head[3], n_eval);
      break;
    }
    // image of the row: last b with gt_off[b] <= gr
    int lo = 0, hi = P.B;
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (__ldg(P.gt_off + mid) <= gr) lo = mid; else hi = mid;
    }
    const int img = lo, g0 = __ldg(P.gt_off + img);
    const int T = __ldg(P.gt_off + img + 1) - g0, t = gr - g0;
    if (t < 0 || t >= T || T > P.max_gt || T > A) continue;   // malformed offsets / flagged images: no rows
    Corners<R> g;
    float4 gb;
    float galo;
    {
      TG cx, cy, w, h;
      Vec4<TG>::load(P.gt_boxes, gr, cx, cy, w, h);
      const Corners<TG> c = corners_of<TG>(cx, cy, w, h);
      g.x1 = (R)c.x1; g.y1 = (R)c.y1; g.x2 = (R)c.x2; g.y2 = (R)c.y2; g.area = (R)c.area;
      const bool ok = finite4((double)g.x1, (double)g.y1, (double)g.x2, (double)g.y2) && isfinite((double)g.area);
      gb = make_float4(f_down((double)g.x1), f_down((double)g.y1), f_up((double)g.x2), f_up((double)g.y2));
      galo = ok ? f_down((double)g.area) : CUDART_NAN_F;
    }
    Cand* cand = P.ws_cand + (size_t)img * kCandCap;
    u64 best_key = 0ull;
    int best_a = 0x7fffffff;
    float rowlo = 0.f;
    u32 rowhi = 0u;
    // exact evaluation of one tile for this row (all lanes)
    auto evaluate = [&](int tile) {
      ++n_eval;
      const int slot = (tile << 5) + lane;
      const int a = P.perm ? __ldg(P.perm + slot) : slot;
      const bool valid = a >= 0 && a < A;
      u64 key = 0ull;
      if (valid) {
        Corners<R> p;
        TP dx, dy, dw, dh;
        Vec4<TP>::load(P.pprior ? P.pprior : P.priors, P.pprior ? slot : a, dx, dy, dw, dh);
        const Corners<TP> c = corners_of<TP>(dx, dy, dw, dh);
        p.x1 = (R)c.x1; p.y1 = (R)c.y1; p.x2 = (R)c.x2; p.y2 = (R)c.y2; p.area = (R)c.area;
        key = key64((double)iou_corners<R>(g, p, EPS));
      }
      const bool listed = key > thr_key;   // phase-2 candidate; one counter update per warp
      const u32 lm = __ballot_sync(SSDG_FULL, listed);
      if (lm) {
        const int leader = __ffs(lm) - 1;
        int base = 0;
        if (lane == leader) base = (int)atomicAdd(&P.ws_ncand[img], (u32)__popc(lm));
        base = __shfl_sync(SSDG_FULL, base, leader);
        if (listed) {
          const int pos = base + __popc(lm & ((1u << lane) - 1u));
          if (pos < kCandCap) { Cand c; c.key = key; c.a = a; c.t = t; cand[pos] = c; }
        }
      }
      // every lane keeps its own best (key, then lowest prior): one arg-max across the warp per ROW.  The running
      // row maximum only prunes: a lower bound of it (the key's high word, one REDUX) is all pass 2 needs.
      if (valid && (key > best_key || (key == best_key && a < best_a))) { best_key = key; best_a = a; }
      const u32 mhi = __reduce_max_sync(SSDG_FULL, (u32)(key >> 32));
      if (mhi > rowhi) {
        rowhi = mhi;
        rowlo = fmaxf(f_down(unkey64((u64)mhi << 32)), 0.f);
      }
    };
    auto tile_ub = [&](const TileStat& ts) {
      float iub, dlb;
      iou_bound(gb, galo, ts, iub, dlb);
      return (ts.safe && dlb > 0.f) ? __fdividef(iub, dlb) * 1.0002f : CUDART_INF_F;   // always > 0
    };
    if (kHier) {
      // Two levels.  A ground-truth box can reach min(thresh, its row maximum) only in a handful of the ~300 tiles, and
      // tiles are ordered shape by shape, block by block: bounding kSuper consecutive tiles at once (their joint
      // statistics) discards most of them in one test.  Lane l keeps the bounds of super-tiles l, 32 + l, ... in registers.
      const int nsuper = (ntiles + kSuper - 1) / kSuper;
      float sub[kSuperRegs];
      float smax = -1.f;
      int sbest = 0x7fffffff;
#pragma unroll
      for (int q = 0; q < kSuperRegs; ++q) {
        const int sp = q * 32 + lane;
        sub[q] = -1.f;                          // < 0: nothing pending
        if (sp < nsuper) {
          sub[q] = tile_ub(P.supers[sp]);
          if (sub[q] > smax) { smax = sub[q]; sbest = sp; }
        }
      }
      {
        const u32 m = __reduce_max_sync(SSDG_FULL, key32(smax));
        sbest = (int)__reduce_min_sync(SSDG_FULL, key32(smax) == m ? (u32)sbest : 0x7fffffffu);
      }
      // the member tile with the highest bound of the best super-tile seeds the running maximum
      int stile;
      {
        const int tile = sbest * kSuper + (lane & (kSuper - 1));
        const float ub = (lane < kSuper && tile < ntiles) ? tile_ub(tiles[tile]) : -1.f;
        const u32 m = __reduce_max_sync(SSDG_FULL, key32(ub));
        stile = (int)__reduce_min_sync(SSDG_FULL, key32(ub) == m ? (u32)tile : 0x7fffffffu);
      }
      evaluate(stile);
      // every super-tile whose bound still reaches min(thresh, running maximum): its members, same test
#pragma unroll
      for (int q = 0; q < kSuperRegs; ++q) {
        if (q * 32 >= nsuper) break;
        for (;;) {
          const bool reach = sub[q] >= 0.f && !(sub[q] < fminf(thr_lo, rowlo));
          const u32 m = __ballot_sync(SSDG_FULL, reach);
          if (!m) break;
          const int l = __ffs(m) - 1;
          if (lane == l) sub[q] = -1.f;
          const int tile = (q * 32 + l) * kSuper + (lane & (kSuper - 1));
          float ub = (lane < kSuper && tile < ntiles && tile != stile) ? tile_ub(tiles[tile]) : -1.f;
          for (;;) {
            const bool r2 = ub >= 0.f && !(ub < fminf(thr_lo, rowlo));
            const u32 m2 = __ballot_sync(SSDG_FULL, r2);
            if (!m2) break;
            const int l2 = __ffs(m2) - 1;
            if (lane == l2) ub = -1.f;
            evaluate((q * 32 + l) * kSuper + l2);
          }
        }
      }
    } else {
    // pass 1: bound every tile; the highest bound seeds the running maximum
    float sub = -1.f;
    int stile = 0x7fffffff;
#pragma unroll 4
    for (int tb = 0; tb < ntiles; tb += 32) {
      const int tile = tb + lane;
      if (tile < ntiles) {
        const float ub = tile_ub(tiles[tile]);
        if (ub > sub) { sub = ub; stile = tile; }
      }
    }
    {
      const u32 m = __reduce_max_sync(SSDG_FULL, key32(sub));
      stile = (int)__reduce_min_sync(SSDG_FULL, key32(sub) == m ? (u32)stile : 0x7fffffffu);
    }
    __syncwarp();
    evaluate(stile);
    // pass 2: every other tile whose bound still reaches min(thresh, running maximum)
    for (int tb = 0; tb < ntiles; tb += 32) {
      const int tile = tb + lane;
      bool pending = tile < ntiles && tile != stile;
      TileStat ts;
      ts.x1 = ts.y1 = ts.x2 = ts.y2 = ts.wmax = ts.hmax = ts.amin = ts.cx1 = ts.cy1 = ts.cx2 = ts.cy2 = 0.f; ts.safe = 1u;
      if (pending) ts = tiles[tile];
      for (;;) {
        const float bound = fminf(thr_lo, rowlo);
        const bool reach = pending && may_reach(gb, galo, ts, bound);
        const u32 m = __ballot_sync(SSDG_FULL, reach);
        if (!m) break;
        const int l = __ffs(m) - 1;
        if (lane == l) pending = false;
        evaluate(tb + l);
      }
    }
    }
    warp_argmax_u64(best_key, best_a);
    if (lane == 0) {
      P.ws_rowkey[(size_t)img * P.tm + t] = best_key;
      P.ws_rowcol[(size_t)img * P.tm + t] = best_a;
    }
    __syncwarp();
  }
}

enum { C_IMG = 0, C_NCAND, C_NRS, C_DONE, C_ROUND, C_DEGEN, C_MINELIM, C_NEXTROW, C_RLO, C_RA, C_RKEY_LO, C_RKEY_HI, C_GENERIC, C_HEAD, C_NLIVE };

template <typename TG, typename TP>
__global__ void __launch_bounds__(kMatchThreads, kMatchCtasPerSm) match_kernel(MatchParams P) {
  typedef typename Promote<TG, TP>::type R;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  MatchSmem<TG, TP> S;
  const bool tiles_in_smem = P.ntiles <= kTileSmemMax;
  S.carve(smem_raw, P.tm, tiles_in_smem ? P.ntiles : 0, P.bits_in_smem ? P.elim_words : 0);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int A = P.A;
  const int ntiles = P.ntiles;
  const R EPS = (R)1e-10;
  const TileStat* tiles = tiles_in_smem ? S.tiles_s : P.tiles;
  u32* elim = P.bits_in_smem ? S.elim_s : P.ws_bits + (size_t)blockIdx.x * 2 * P.elim_words;
  u32* touch = P.bits_in_smem ? S.touch_s : elim + P.elim_words;
  u64* colkey = P.ws_colkey + (size_t)blockIdx.x * A;
  int* colt = P.ws_colt + (size_t)blockIdx.x * A;
  const u64 thr_key = key64((double)(R)P.thresh);
  const float thr_lo = f_down((double)(R)P.thresh);

  // once per CTA: stage the tile statistics, clear the column scratch
  if (tiles_in_smem)
    for (int i = tid; i < ntiles; i += kMatchThreads) S.tiles_s[i] = P.tiles[i];
  for (int a = tid; a < A; a += kMatchThreads) { colkey[a] = 0ull; colt[a] = 0x7fffffff; }

  auto load_prior = [&](int a, Corners<R>& p, TP& dx, TP& dy, TP& dw, TP& dh) {
    Vec4<TP>::load(P.priors, a, dx, dy, dw, dh);
    Corners<TP> c = corners_of<TP>(dx, dy, dw, dh);
    p.x1 = (R)c.x1; p.y1 = (R)c.y1; p.x2 = (R)c.x2; p.y2 = (R)c.y2; p.area = (R)c.area;
  };
  auto load_gt = [&](int t) {
    Corners<R> g;
    g.x1 = S.gx1[t]; g.y1 = S.gy1[t]; g.x2 = S.gx2[t]; g.y2 = S.gy2[t]; g.area = S.ga[t];
    return g;
  };
  auto bit_test = [&](const u32* bm, int a) { return (bm[a >> 5] >> (a & 31)) & 1u; };

  // The index must belong to THESE priors (in-place edits such as ssdg_priors_clip, or a recycled address, would
  // silently pair with stale tiles): one CTA re-derives the content checksum and raises status bit 3 on mismatch.
  if (P.index_sum != 0ull && blockIdx.x == 0) {
    const u64* w = reinterpret_cast<const u64*>(P.priors);
    u64 acc = 0ull;
    for (long long i = tid; i < P.prior_words; i += kMatchThreads) acc += checksum_term(__ldg(w + i), i);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(SSDG_FULL, acc, o);
    u64* cs = reinterpret_cast<u64*>(&S.ctl[C_RKEY_LO]);   // 8-byte aligned pair of control words (free before the loop)
    if (tid == 0) *cs = 0ull;
    __syncthreads();
    if (lane == 0) atomicAdd(reinterpret_cast<unsigned long long*>(cs), (unsigned long long)acc);
    __syncthreads();
    if (tid == 0 && *cs != P.index_sum) atomicOr(&P.ws_head[1], 8u);
    __syncthreads();
  }

  // everything above is independent of the row search: launched as its programmatic dependent, the CTAs do it while
  // the search drains, and only now wait for its results
  pdl_wait();
#ifdef SSDG_MATCH_TIMING
  long long tk0 = 0;
#define TICK(slot) do { __syncthreads(); if (tid == 0) { long long n_ = clock64(); atomicAdd((unsigned long long*)&P.ws_head[8 + 2 * (slot)], (unsigned long long)(n_ - tk0)); tk0 = n_; } } while (0)
#else
#define TICK(slot) do { } while (0)
#endif
  for (;;) {
    __syncthreads();
#ifdef SSDG_MATCH_TIMING
    if (tid == 0) tk0 = clock64();
#endif
    if (tid == 0) S.ctl[C_IMG] = (int)atomicAdd(&P.ws_head[0], 1u);
    __syncthreads();
    const int img = S.ctl[C_IMG];
    if (img >= P.B) break;
    const int g0 = P.gt_off[img];
    int T = P.gt_off[img + 1] - g0;
    if (T < 0) T = 0;
    bool bad = false;
    if (T > P.max_gt) { if (tid == 0) atomicOr(&P.ws_head[1], 1u); bad = true; }
    if (T > A) { if (tid == 0) atomicOr(&P.ws_head[1], 2u); bad = true; }
    if (bad) T = 0;  // outputs for the image are still fully written (all unmatched)
    const size_t obase = (size_t)img * A;
    const Cand* cand = P.ws_cand + (size_t)img * kCandCap;

    // ---- per-image setup -------------------------------------------------------------------
    for (int t = tid; t < T; t += kMatchThreads) {
      TG cx, cy, w, h;
      Vec4<TG>::load(P.gt_boxes, g0 + t, cx, cy, w, h);
      Corners<TG> c = corners_of<TG>(cx, cy, w, h);
      R x1 = (R)c.x1, y1 = (R)c.y1, x2 = (R)c.x2, y2 = (R)c.y2, ar = (R)c.area;
      S.gx1[t] = x1; S.gy1[t] = y1; S.gx2[t] = x2; S.gy2[t] = y2; S.ga[t] = ar;
      const bool ok = finite4((double)x1, (double)y1, (double)x2, (double)y2) && isfinite((double)ar);
      S.cbox[t] = make_float4(f_down((double)x1), f_down((double)y1), f_up((double)x2), f_up((double)y2));
      S.galo[t] = ok ? f_down((double)ar) : CUDART_NAN_F;
      S.rowkey[t] = P.ws_rowkey[(size_t)img * P.tm + t];     // the search kernel's result for this row
      S.rowcol[t] = P.ws_rowcol[(size_t)img * P.tm + t];
      S.dead[t] = 0;
    }
    for (int w = tid; w < P.elim_words; w += kMatchThreads) { elim[w] = 0u; touch[w] = 0u; }
    if (tid == 0) {
      S.ctl[C_NCAND] = 0; S.ctl[C_NRS] = 0; S.ctl[C_DONE] = 0; S.ctl[C_ROUND] = 0; S.ctl[C_DEGEN] = 0;
      S.ctl[C_MINELIM] = 0x7fffffff; S.ctl[C_NEXTROW] = 0; S.ctl[C_GENERIC] = 0; S.ctl[C_HEAD] = 0; S.ctl[C_NLIVE] = -1;
    }
    __syncthreads();

    TICK(0);
    // Re-search of ONE row over the live columns by the whole CTA (a row whose cached column was taken):
    // the warps split the tiles, share the running maximum through shared memory, and the first
    // arg-max column is settled after a barrier.  Same exact evaluation, same bound, just parallel.
    auto research_row = [&](int t) {
      u64* skey = reinterpret_cast<u64*>(&S.ctl[C_RKEY_LO]);   // 8-byte aligned pair of control words
      if (tid == 0) { *skey = 0ull; S.ctl[C_RA] = 0x7fffffff; S.ctl[C_RLO] = 0; }
      __syncthreads();
      const Corners<R> g = load_gt(t);
      const float4 gb = S.cbox[t];
      const float galo = S.galo[t];
      u64 my_key = 0ull;
      int my_a = 0x7fffffff;
      for (int tb = warp * 32; tb < ntiles; tb += (kMatchThreads / 32) * 32) {
        const int tile = tb + lane;
        bool pending = tile < ntiles;
        float ub = 0.f;
        if (pending) {
          const TileStat ts = tiles[tile];
          float iub, dlb;
          iou_bound(gb, galo, ts, iub, dlb);
          ub = (ts.safe && dlb > 0.f) ? __fdividef(iub, dlb) * 1.0002f : CUDART_INF_F;
        }
        for (;;) {
          const float rowlo = __int_as_float(*reinterpret_cast<volatile int*>(&S.ctl[C_RLO]));
          const bool reach = pending && !(ub < fminf(thr_lo, rowlo));
          if (!__ballot_sync(SSDG_FULL, reach)) break;
          // highest bound first
          const u32 mk = __reduce_max_sync(SSDG_FULL, reach ? key32(ub) : 0u);
          const int l = __ffs(__ballot_sync(SSDG_FULL, reach && key32(ub) == mk)) - 1;
          if (lane == l) pending = false;
          const int slot = ((tb + l) << 5) + lane;
          const int a = P.perm ? __ldg(P.perm + slot) : slot;
          const bool valid = a >= 0 && a < A && !bit_test(elim, a);
          u64 key = 0ull;
          if (valid) {
            Corners<R> p; TP dx, dy, dw, dh;
            if (P.pprior) {
              Vec4<TP>::load(P.pprior, slot, dx, dy, dw, dh);
              Corners<TP> c = corners_of<TP>(dx, dy, dw, dh);
              p.x1 = (R)c.x1; p.y1 = (R)c.y1; p.x2 = (R)c.x2; p.y2 = (R)c.y2; p.area = (R)c.area;
            } else {
              load_prior(a, p, dx, dy, dw, dh);
            }
            key = key64((double)iou_corners<R>(g, p, EPS));
          }
          u64 wk = key;
          int wa = valid ? a : 0x7fffffff;
          warp_argmax_u64(wk, wa);
          if (wk > my_key || (wk == my_key && wa < my_a)) { my_key = wk; my_a = wa; }
          if (lane == 0 && wk > 0ull) {
            atomicMax(skey, wk);
            atomicMax(&S.ctl[C_RLO], __float_as_int(fmaxf(f_down(unkey64(wk)), 0.f)));
          }
        }
      }
      __syncthreads();
      if (lane == 0 && my_key == *skey && my_key != 0ull) atomicMin(&S.ctl[C_RA], my_a);
      __syncthreads();
      if (tid == 0) { S.rowkey[t] = *skey; S.rowcol[t] = S.ctl[C_RA]; }
      __syncthreads();
    };

    TICK(1);

    // ---- phase 2: first-arg-max row of every listed prior ---------------------------------------------
    const int ncand_raw = bad ? 0 : (int)P.ws_ncand[img];
    const bool cand_overflow = ncand_raw > kCandCap;
    const int ncand = cand_overflow ? 0 : ncand_raw;
    if (cand_overflow) {
      // more pairs above the threshold than the list holds: exhaustive exact scan, one prior per thread
      if (tid == 0) atomicOr(&P.ws_head[1], 4u);
      for (int a = tid; a < A; a += kMatchThreads) {
        Corners<R> p; TP dx, dy, dw, dh;
        load_prior(a, p, dx, dy, dw, dh);
        u64 bk = 0ull;
        int bt = 0x7fffffff;
        for (int t = 0; t < T; ++t) {
          const u64 k = key64((double)iou_corners<R>(load_gt(t), p, EPS));
          if (k > bk) { bk = k; bt = t; }
        }
        if (bk > thr_key) { colkey[a] = bk; colt[a] = bt; atomicOr(&touch[a >> 5], 1u << (a & 31)); }
      }
    } else {
      for (int e = tid; e < ncand; e += kMatchThreads) {
        const Cand c = cand[e];
        atomicMax(&colkey[c.a], c.key);
        atomicOr(&touch[c.a >> 5], 1u << (c.a & 31));
      }
      __syncthreads();
      for (int e = tid; e < ncand; e += kMatchThreads) {
        const Cand c = cand[e];
        if (c.key == colkey[c.a]) atomicMin(&colt[c.a], c.t);
      }
    }
    __syncthreads();

    TICK(2);
    // ---- greedy rounds (utils/bbox.py:62-68) --------------------------------------------------------
    if (T > 0)
    for (;;) {
      // Fast path.  The global arg-max of a round is the row with the largest cached maximum, so the
      // rounds walk the rows in descending (key, then ascending row) order -- a priority queue with lazy
      // re-evaluation: a row whose cached column has been taken in the meantime only gives an upper
      // bound, so it is re-searched (with every other stale row) and the order is rebuilt.
      const bool fast = !S.ctl[C_GENERIC];
      if (fast && S.ctl[C_NLIVE] < 0) {
        // (re)build the order of the live rows by rank counting: one warp per row, lanes split the others
        for (int t = warp; t < T; t += kMatchThreads / 32) {
          if (S.dead[t]) continue;
          const u64 kt = S.rowkey[t];
          int cnt = 0;
          for (int u = lane; u < T; u += 32)
            if (!S.dead[u]) { const u64 ku = S.rowkey[u]; cnt += (ku > kt || (ku == kt && u < t)) ? 1 : 0; }
          cnt = (int)__reduce_add_sync(SSDG_FULL, (u32)cnt);
          if (lane == 0) S.order[cnt] = t;
        }
        if (warp == 0) {
          int nl = 0;
          for (int u = lane; u < T; u += 32) nl += S.dead[u] ? 0 : 1;
          nl = (int)__reduce_add_sync(SSDG_FULL, (u32)nl);
          if (lane == 0) { S.ctl[C_NLIVE] = nl; S.ctl[C_HEAD] = 0; }
        }
        __syncthreads();
      }
      if (warp == 0 && fast) {
        int round = S.ctl[C_ROUND];
        int head = S.ctl[C_HEAD];
        const int nlive = S.ctl[C_NLIVE];
        int nrs = 0;
        bool stop = false;
        // 32 queue positions per step: all positions before the first stale one are taken at once
        while (!stop && head < nlive && round < T) {
          const int p = head + lane;
          const bool in = p < nlive && (round + lane) < T;
          int t = 0, a = 0;
          u64 k = ~0ull;
          if (in) { t = S.order[p]; k = S.rowkey[t]; a = S.rowcol[t]; }
          const bool degen_here = in && k <= SSDG_KEY_ZERO && (round + lane) > 0;
          const u32 same = __match_any_sync(SSDG_FULL, in ? a : -1 - lane);
          const bool stale = in && (bit_test(elim, a) || (same & ((1u << lane) - 1u)) != 0u);
          const u32 bad = __ballot_sync(SSDG_FULL, stale || degen_here || !in);
          const int ntake = bad ? __ffs(bad) - 1 : 32;
          if (lane < ntake) {
            S.pair_t[round + lane] = t;
            S.pair_a[round + lane] = a;
            S.dead[t] = 1;
            atomicOr(&elim[a >> 5], 1u << (a & 31));
            atomicMin(&S.ctl[C_MINELIM], a);
          }
          __syncwarp();
          round += ntake; head += ntake;
          if (ntake < 32) {
            const u32 dg = __ballot_sync(SSDG_FULL, degen_here);
            const u32 st = __ballot_sync(SSDG_FULL, stale);
            if (dg && (__ffs(dg) - 1) == ntake) { if (lane == 0) S.ctl[C_GENERIC] = 1; stop = true; }
            else if (st && (__ffs(st) - 1) == ntake) stop = true;
          }
        }
        if (stop && round < T) {
          // every live row whose cached column is gone is re-searched now; the order is rebuilt afterwards
          __syncwarp();
          for (int r = 0; r * 32 < T; ++r) {
            const int t = lane + 32 * r;
            const bool need = t < T && !S.dead[t] && bit_test(elim, S.rowcol[t]);
            const u32 nm = __ballot_sync(SSDG_FULL, need);
            if (need) S.rs_list[nrs + __popc(nm & ((1u << lane) - 1u))] = t;
            nrs += __popc(nm);
          }
          if (lane == 0) S.ctl[C_NLIVE] = -1;
        }
        if (lane == 0) { S.ctl[C_ROUND] = round; S.ctl[C_HEAD] = head; S.ctl[C_NRS] = nrs; S.ctl[C_DONE] = round >= T; }
      } else if (warp == 0) {
        int round = S.ctl[C_ROUND];
        int nrs = 0;
        while (round < T) {
          u64 bk = 0ull;
          int bt = 0x7fffffff;
          for (int t = lane; t < T; t += 32) {
            if (!S.dead[t]) {
              u64 k = S.rowkey[t];
              if (k > bk) { bk = k; bt = t; }
            }
          }
          warp_argmax_u64(bk, bt);
          int wt, wa;
          if (bk > SSDG_KEY_ZERO || round == 0) {
            wt = bt;
            wa = S.rowcol[bt];
          } else {
            if (lane == 0) {
              u64 best = 0ull;
              long long bflat = 0x7fffffffffffffffll;
              const int me = S.ctl[C_MINELIM];
              for (int t = 0; t < T; ++t) {
                u64 k; long long f;
                if (S.dead[t]) { k = SSDG_KEY_ZERO; f = (long long)t * A; }
                else {
                  k = S.rowkey[t]; f = (long long)t * A + S.rowcol[t];
                  if (k > best || (k == best && f < bflat)) { best = k; bflat = f; }
                  k = SSDG_KEY_ZERO; f = (long long)t * A + me;
                }
                if (k > best || (k == best && f < bflat)) { best = k; bflat = f; }
              }
              S.red_idx[0] = (int)(bflat / A);
              S.red_idx[1] = (int)(bflat % A);
              S.ctl[C_DEGEN] = 1;
            }
            __syncwarp();
            wt = S.red_idx[0];
            wa = S.red_idx[1];
          }
          const bool fresh = !bit_test(elim, wa);
          __syncwarp();
          if (lane == 0) {
            S.pair_t[round] = wt;
            S.pair_a[round] = wa;
            S.dead[wt] = 1;
            elim[wa >> 5] |= 1u << (wa & 31);
            if (wa < S.ctl[C_MINELIM]) S.ctl[C_MINELIM] = wa;
          }
          __syncwarp();
          ++round;
          if (fresh && round < T) {
            for (int t0 = 0; t0 < T; t0 += 32) {
              const int t = t0 + lane;
              const bool need = t < T && !S.dead[t] && S.rowcol[t] == wa;
              const u32 nm = __ballot_sync(SSDG_FULL, need);
              if (need) S.rs_list[nrs + __popc(nm & ((1u << lane) - 1u))] = t;
              nrs += __popc(nm);
            }
          }
          if (nrs > 0) break;
        }
        if (lane == 0) { S.ctl[C_ROUND] = round; S.ctl[C_NRS] = nrs; S.ctl[C_DONE] = round >= T; }
      }
      __syncthreads();
      const int nrs = S.ctl[C_NRS];
      const bool done = S.ctl[C_DONE] != 0;
      if (done && nrs == 0) break;
#ifdef SSDG_MATCH_TIMING
      if (tid == 0 && nrs > 0) { atomicAdd(&P.ws_head[40], 1u); atomicAdd(&P.ws_head[41], (u32)nrs); }
      long long rs0 = clock64();
#endif
      for (int i = 0; i < nrs; ++i) research_row(S.rs_list[i]);
#ifdef SSDG_MATCH_TIMING
      if (tid == 0 && nrs > 0) atomicAdd((unsigned long long*)&P.ws_head[42], (unsigned long long)(clock64() - rs0));
#endif
      __syncthreads();
      if (tid == 0) { S.ctl[C_NRS] = 0; S.ctl[C_NEXTROW] = 0; }
      __syncthreads();
      if (done) break;
    }

    TICK(3);
    // ---- output: every prior once, in prior order (phase 2), then the phase-1 pairs ---------------------
    auto emit_prior = [&](int a, bool pos, const float4& un) {
      float bx = 0.f, by = 0.f, bw = 0.f, bh = 0.f;
      int lab = 0, ct = -1;
      if (pos) {
        ct = colt[a];
        TG gx, gy, gw, gh;
        Vec4<TG>::load(P.gt_boxes, g0 + ct, gx, gy, gw, gh);
        bx = (float)gx; by = (float)gy; bw = (float)gw; bh = (float)gh;
        lab = (int)__ldg(P.gt_cls + g0 + ct);
        colkey[a] = 0ull; colt[a] = 0x7fffffff;     // leave the scratch clean for the next image
      }
      if (P.out_cls) P.out_cls[obase + a] = lab;
      if (P.out_mask) P.out_mask[obase + a] = pos ? 1 : 0;
      if (P.out_match) P.out_match[obase + a] = ct;
      if (P.out_box) reinterpret_cast<float4*>(P.out_box)[obase + a] = make_float4(bx, by, bw, bh);
      if (P.out_loc) {
        float4 enc = un;
        if (pos || !P.unmatched) {
          TP dx, dy, dw, dh;
          Vec4<TP>::load(P.priors, a, dx, dy, dw, dh);
          enc = encode_row<TP>(bx, by, bw, bh, dx, dy, dw, dh);
        }
        reinterpret_cast<float4*>(P.out_loc)[obase + a] = enc;
      }
    };
    {
      // Positives are ~3 % of the priors and their encoding is ~300 float64 instructions (two logarithms, four
      // divisions): inside the prior-order sweep nearly every warp would run that path for one or two lanes.  So the
      // sweep writes every prior as unmatched, and the positives are then taken DENSELY from the image's pair list
      // (the entry that won its column: maximum key, then lowest row).  With an overflown list the sweep decides by
      // the touch bits as before.
      const bool dense_pos = !cand_overflow;
      const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
      int a = tid;
      for (; a + 3 * kMatchThreads < A; a += 4 * kMatchThreads) {   // four independent priors per iteration
        float4 u[4];
        bool p4[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int aq = a + q * kMatchThreads;
          p4[q] = !dense_pos && bit_test(touch, aq) != 0;
          u[q] = (P.unmatched && P.out_loc) ? __ldg(P.unmatched + aq) : z4;
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) emit_prior(a + q * kMatchThreads, p4[q], u[q]);
      }
      for (; a < A; a += kMatchThreads)
        emit_prior(a, !dense_pos && bit_test(touch, a) != 0, (P.unmatched && P.out_loc) ? __ldg(P.unmatched + a) : z4);
      if (dense_pos) {
        __syncthreads();
        for (int e = tid; e < ncand; e += kMatchThreads) {
          const Cand c = cand[e];
          if (c.key == colkey[c.a] && c.t == colt[c.a]) emit_prior(c.a, true, z4);
        }
      }
    }
    __syncthreads();
    // phase-1 pairs (utils/bbox.py:87-90; later pairs win)
    const bool degen = S.ctl[C_DEGEN] != 0;
    for (int k = tid; k < T; k += kMatchThreads) {
      const int t = S.pair_t[k], a = S.pair_a[k];
      bool last = true;
      if (degen)
        for (int k2 = k + 1; k2 < T; ++k2)
          if (S.pair_a[k2] == a) { last = false; break; }
      if (!last) continue;
      TG gx, gy, gw, gh;
      Vec4<TG>::load(P.gt_boxes, g0 + t, gx, gy, gw, gh);
      const float bx = (float)gx, by = (float)gy, bw = (float)gw, bh = (float)gh;
      if (P.out_cls) P.out_cls[obase + a] = (int)__ldg(P.gt_cls + g0 + t);
      if (P.out_mask) P.out_mask[obase + a] = 1;
      if (P.out_match) P.out_match[obase + a] = t;
      if (P.out_box) reinterpret_cast<float4*>(P.out_box)[obase + a] = make_float4(bx, by, bw, bh);
      if (P.out_loc) {
        TP dx, dy, dw, dh;
        Vec4<TP>::load(P.priors, a, dx, dy, dw, dh);
        reinterpret_cast<float4*>(P.out_loc)[obase + a] = encode_row<TP>(bx, by, bw, bh, dx, dy, dw, dh);
      }
    }
    TICK(4);
  }
}

template <typename TG, typename TP>
static int launch_match(const MatchParams& P, int grid, size_t smem, cudaStream_t st) {
  if (!P.perm) {
    tile_stats_kernel<TP><<<(P.ntiles * 32 + 255) / 256, 256, 0, st>>>(P.priors, P.A, nullptr, P.ntiles,
                                                                       const_cast<TileStat*>(P.tiles));
    const int nsuper = (P.ntiles + kSuper - 1) / kSuper;
    super_stats_kernel<<<(nsuper + 127) / 128, 128, 0, st>>>(P.tiles, P.ntiles, const_cast<TileStat*>(P.supers));
    SSDG_LAUNCH_CHECK();
  }
  if (smem > 48 * 1024)
    SSDG_CUDA_TRY(cudaFuncSetAttribute(match_kernel<TG, TP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // same shared-memory carve-out as the streaming kernels so CTAs of both can share an SM
  SSDG_CUDA_TRY(cudaFuncSetAttribute(match_kernel<TG, TP>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  prof_begin(SSDG_PROF_MATCH, st);
  {
    const bool hier = P.ntiles <= kTileSmemMax;
    const size_t ssm = 0;
    auto skern = hier ? search_kernel<TG, TP, true> : search_kernel<TG, TP, false>;
    SSDG_CUDA_TRY(cudaFuncSetAttribute(skern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    long long sgrid = (long long)sm_count() * kSearchCtasPerSm;
    const long long want = ((long long)P.B * (P.max_gt > 0 ? P.max_gt : 1) + kSearchWarps - 1) / kSearchWarps;
    if (want < sgrid) sgrid = want;
    prof_begin(SSDG_PROF_SEARCH, st);
    skern<<<(unsigned)sgrid, kSearchThreads, ssm, st>>>(P);
    prof_end(SSDG_PROF_SEARCH, st);
    SSDG_LAUNCH_CHECK();
  }
  SSDG_CUDA_TRY(launch_pdl(match_kernel<TG, TP>, dim3(grid), dim3(kMatchThreads), smem, st, P));
  prof_end(SSDG_PROF_MATCH, st);
  SSDG_LAUNCH_CHECK();
  return SSDG_OK;
}

static int match_ws_ctas(int batch) { return batch < kMatchMaxCtas ? batch : kMatchMaxCtas; }
static int match_grid(int batch) {
  int g = sm_count() * kMatchCtasPerSm;
  if (g > kMatchMaxCtas) g = kMatchMaxCtas;
  return batch < g ? batch : g;
}

struct MatchWs {
  u32* head;
  u32* ncand;
  u64* rowkey;
  int* rowcol;
  Cand* cand;
  u64* colkey;
  int* colt;
  u32* bits;
  TileStat* tiles;
  TileStat* supers;
};
static int match_tm(int max_gt) {
  const int tm = ((max_gt + 31) / 32) * 32;
  return tm == 0 ? 32 : tm;
}
static size_t match_ws_layout(int batch, int n_priors, int max_gt, int ctas, MatchWs* out, unsigned char* base) {
  size_t o = 0;
  const size_t words = ((size_t)n_priors + 31) / 32;
  const size_t rows = (size_t)batch * match_tm(max_gt);
  if (out) out->head = (u32*)(base + o);
  o += 256;
  if (out) out->ncand = (u32*)(base + o);          // directly behind the head: cleared by the same memset
  o += align_up((size_t)batch * 4, 256);
  if (out) out->rowkey = (u64*)(base + o);
  o += align_up(rows * 8, 256);
  if (out) out->rowcol = (int*)(base + o);
  o += align_up(rows * 4, 256);
  if (out) out->cand = (Cand*)(base + o);
  o += align_up((size_t)batch * kCandCap * sizeof(Cand), 256);
  if (out) out->colkey = (u64*)(base + o);
  o += align_up((size_t)ctas * n_priors * 8, 256);
  if (out) out->colt = (int*)(base + o);
  o += align_up((size_t)ctas * n_priors * 4, 256);
  if (out) out->bits = (u32*)(base + o);
  o += align_up((size_t)ctas * 2 * words * 4, 256);
  if (out) out->tiles = (TileStat*)(base + o);
  o += align_up(words * sizeof(TileStat), 256);
  if (out) out->supers = (TileStat*)(base + o);
  o += align_up((words / kSuper + 1) * sizeof(TileStat), 256);
  return o;
}

// ---- prior index ---------------------------------------------------------------------------------------
constexpr int kIndexMaxShapes = 64;
struct IndexInfo { int n_priors, ntiles, dtype, device; u64 sum; };
static std::mutex g_index_mu;
static std::unordered_map<const void*, IndexInfo> g_index;   // index device pointer -> geometry, owner device, checksum
                                                             // (erased by ssdg_prior_index_destroy)

static size_t index_slots(int n_priors) { return ((size_t)n_priors + 31) / 32 * 32 + (size_t)kIndexMaxShapes * 32; }
static size_t index_perm_offset() { return 256; }
static size_t index_tiles_offset(int n_priors) { return 256 + align_up(index_slots(n_priors) * 4, 256); }
static size_t index_supers_offset(int n_priors) {
  return index_tiles_offset(n_priors) + align_up(index_slots(n_priors) / 32 * sizeof(TileStat), 256);
}
static size_t index_unmatched_offset(int n_priors) {
  return index_supers_offset(n_priors) + align_up((index_slots(n_priors) / 32 / kSuper + 1) * sizeof(TileStat), 256);
}
static size_t index_pprior_offset(int n_priors) { return index_unmatched_offset(n_priors) + align_up((size_t)n_priors * 16, 256); }

}  // namespace ssdg

using namespace ssdg;

extern "C" size_t ssdg_prior_index_bytes(int32_t n_priors) {
  if (n_priors <= 0) return 0;
  return index_pprior_offset(n_priors) + align_up(index_slots(n_priors) * 32, 256);
}

extern "C" int ssdg_prior_index_build(const void* priors, int32_t prior_dtype, int32_t n_priors, void* index,
                                      size_t index_bytes, void* stream) {
  if (!priors || !index || n_priors <= 0) return SSDG_ERR_ARG;
  if (prior_dtype != SSDG_F32 && prior_dtype != SSDG_F64) return SSDG_ERR_ARG;
  if (n_priors >= (1 << kABits)) return SSDG_ERR_LIMIT;
  if (((uintptr_t)index & 255) || index_bytes < ssdg_prior_index_bytes(n_priors)) return SSDG_ERR_WORKSPACE;
  if ((uintptr_t)priors & 15) return SSDG_ERR_ALIGN;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t esz = prior_dtype == SSDG_F64 ? 8 : 4;
  std::vector<unsigned char> raw((size_t)n_priors * 4 * esz);
  SSDG_CUDA_TRY(cudaMemcpyAsync(raw.data(), priors, raw.size(), cudaMemcpyDeviceToHost, st));
  SSDG_CUDA_TRY(cudaStreamSynchronize(st));
  auto at = [&](int a, int k) -> double {
    return prior_dtype == SSDG_F64 ? reinterpret_cast<const double*>(raw.data())[(size_t)a * 4 + k]
                                   : (double)reinterpret_cast<const float*>(raw.data())[(size_t)a * 4 + k];
  };
  // shape classes: identical (w, h); too many distinct shapes -> one class (spatial blocking only)
  std::map<std::pair<double, double>, int> shape_id;
  std::vector<int> cls(n_priors);
  bool one_class = false;
  for (int a = 0; a < n_priors && !one_class; ++a) {
    auto key = std::make_pair(at(a, 2), at(a, 3));
    auto it = shape_id.find(key);
    if (it == shape_id.end()) {
      if ((int)shape_id.size() >= kIndexMaxShapes) { one_class = true; break; }
      it = shape_id.emplace(key, (int)shape_id.size()).first;
    }
    cls[a] = it->second;
  }
  if (one_class) std::fill(cls.begin(), cls.end(), 0);
  const int ncls = one_class ? 1 : (int)shape_id.size();
  std::vector<std::vector<int>> members(ncls);
  for (int a = 0; a < n_priors; ++a) members[cls[a]].push_back(a);
  std::vector<int> perm;
  perm.reserve(index_slots(n_priors));
  for (auto& mem : members) {
    // block the class into ~32-prior cells of a g x g grid over its centres, row-major blocks
    double x0 = 1e300, x1 = -1e300, y0 = 1e300, y1 = -1e300;
    for (int a : mem) {
      const double cx = at(a, 0), cy = at(a, 1);
      if (cx == cx && cy == cy) { x0 = std::min(x0, cx); x1 = std::max(x1, cx); y0 = std::min(y0, cy); y1 = std::max(y1, cy); }
    }
    int g = 1;
    while ((size_t)g * g * 32 < mem.size()) ++g;
    const double sx = x1 > x0 ? g / (x1 - x0) : 0.0, sy = y1 > y0 ? g / (y1 - y0) : 0.0;
    auto block = [&](int a) {
      const double cx = at(a, 0), cy = at(a, 1);
      int bx = (cx == cx) ? (int)std::min<double>(g - 1, std::max(0.0, (cx - x0) * sx)) : 0;
      int by = (cy == cy) ? (int)std::min<double>(g - 1, std::max(0.0, (cy - y0) * sy)) : 0;
      return by * g + bx;
    };
    std::vector<std::pair<int, int>> keyed;
    keyed.reserve(mem.size());
    for (int a : mem) keyed.emplace_back(block(a), a);
    std::stable_sort(keyed.begin(), keyed.end());
    for (auto& kv : keyed) perm.push_back(kv.second);
    while (perm.size() % 32) perm.push_back(-1);
  }
  const int ntiles = (int)(perm.size() / 32);
  if (perm.size() > index_slots(n_priors)) return SSDG_ERR_LIMIT;
  unsigned char* base = (unsigned char*)index;
  int header[4] = {n_priors, ntiles, 0, 0};
  SSDG_CUDA_TRY(cudaMemcpyAsync(base, header, sizeof(header), cudaMemcpyHostToDevice, st));
  SSDG_CUDA_TRY(cudaMemcpyAsync(base + index_perm_offset(), perm.data(), perm.size() * 4, cudaMemcpyHostToDevice, st));
  {
    // the priors in slot order (padding slots hold a copy of prior 0; they are never valid)
    std::vector<unsigned char> pp(perm.size() * 4 * esz);
    for (size_t sl = 0; sl < perm.size(); ++sl)
      std::copy_n(raw.data() + (size_t)(perm[sl] < 0 ? 0 : perm[sl]) * 4 * esz, 4 * esz, pp.data() + sl * 4 * esz);
    SSDG_CUDA_TRY(cudaMemcpyAsync(base + index_pprior_offset(n_priors), pp.data(), pp.size(), cudaMemcpyHostToDevice, st));
    SSDG_CUDA_TRY(cudaStreamSynchronize(st));
  }
  TileStat* tiles = (TileStat*)(base + index_tiles_offset(n_priors));
  TileStat* supers = (TileStat*)(base + index_supers_offset(n_priors));
  float4* unmatched = (float4*)(base + index_unmatched_offset(n_priors));
  const int* dperm = (const int*)(base + index_perm_offset());
  if (prior_dtype == SSDG_F64) {
    tile_stats_kernel<double><<<(ntiles * 32 + 255) / 256, 256, 0, st>>>(priors, n_priors, dperm, ntiles, tiles);
    unmatched_kernel<double><<<(n_priors + 255) / 256, 256, 0, st>>>(priors, n_priors, unmatched);
  } else {
    tile_stats_kernel<float><<<(ntiles * 32 + 255) / 256, 256, 0, st>>>(priors, n_priors, dperm, ntiles, tiles);
    unmatched_kernel<float><<<(n_priors + 255) / 256, 256, 0, st>>>(priors, n_priors, unmatched);
  }
  super_stats_kernel<<<((ntiles + kSuper - 1) / kSuper + 127) / 128, 128, 0, st>>>(tiles, ntiles, supers);
  SSDG_LAUNCH_CHECK();
  SSDG_CUDA_TRY(cudaStreamSynchronize(st));
  u64 sum = 0ull;
  {
    const u64* w = reinterpret_cast<const u64*>(raw.data());
    const long long nw = (long long)(raw.size() / 8);
    for (long long i = 0; i < nw; ++i) sum += checksum_term(w[i], i);
    if (sum == 0ull) sum = 1ull;   // 0 means "no index" on the device side
  }
  int dev = 0;
  SSDG_CUDA_TRY(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(g_index_mu);
  g_index[index] = IndexInfo{n_priors, ntiles, prior_dtype, dev, sum};
  return SSDG_OK;
}

extern "C" int ssdg_prior_index_destroy(void* index) {
  if (!index) return SSDG_OK;
  std::lock_guard<std::mutex> lk(g_index_mu);
  return g_index.erase(index) ? SSDG_OK : SSDG_ERR_ARG;
}

extern "C" size_t ssdg_match_workspace_bytes(int32_t batch, int32_t n_priors, int32_t max_gt) {
  if (batch <= 0 || n_priors <= 0 || max_gt < 0) return 0;
  if (max_gt > n_priors) max_gt = n_priors;
  return match_ws_layout(batch, n_priors, max_gt, match_ws_ctas(batch), nullptr, nullptr);
}

extern "C" int ssdg_match_encode(const void* gt_boxes, int32_t gt_dtype, const float* gt_cls,
                                 const int32_t* gt_offsets, const void* priors, int32_t prior_dtype,
                                 const void* prior_index, int32_t batch, int32_t n_priors, int32_t max_gt, double thresh,
                                 int32_t* out_cls, float* out_box, float* out_loc, uint8_t* out_mask,
                                 int32_t* out_match, void* workspace, size_t workspace_bytes, void* stream) {
  if (!gt_boxes || !gt_cls || !gt_offsets || !priors || batch <= 0 || n_priors <= 0 || max_gt < 0) return SSDG_ERR_ARG;
  if ((gt_dtype != SSDG_F32 && gt_dtype != SSDG_F64) || (prior_dtype != SSDG_F32 && prior_dtype != SSDG_F64))
    return SSDG_ERR_ARG;
  if (!(thresh > 0.0)) return SSDG_ERR_THRESH;
  if (n_priors >= (1 << kABits) || max_gt > kMaxGT) return SSDG_ERR_LIMIT;
  if (max_gt > n_priors) max_gt = n_priors;  // images with more GT than priors raise status bit 1
  if (((uintptr_t)gt_boxes | (uintptr_t)priors | (uintptr_t)out_box | (uintptr_t)out_loc) & 15) return SSDG_ERR_ALIGN;
  if (!workspace || ((uintptr_t)workspace & 255) || workspace_bytes < ssdg_match_workspace_bytes(batch, n_priors, max_gt))
    return SSDG_ERR_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = match_grid(batch);
  MatchWs ws;
  match_ws_layout(batch, n_priors, max_gt, match_ws_ctas(batch), &ws, (unsigned char*)workspace);
  MatchParams P;
  P.gt_boxes = gt_boxes; P.gt_cls = gt_cls; P.gt_off = gt_offsets; P.priors = priors;
  P.B = batch; P.A = n_priors; P.max_gt = max_gt; P.tm = match_tm(max_gt);
  P.thresh = thresh;
  P.out_cls = out_cls; P.out_box = out_box; P.out_loc = out_loc; P.out_mask = out_mask; P.out_match = out_match;
  P.elim_words = (n_priors + 31) / 32;
  P.ws_head = ws.head; P.ws_ncand = ws.ncand; P.ws_rowkey = ws.rowkey; P.ws_rowcol = ws.rowcol; P.ws_cand = ws.cand; P.ws_colkey = ws.colkey; P.ws_colt = ws.colt; P.ws_bits = ws.bits;
  P.tiles = ws.tiles; P.supers = ws.supers; P.perm = nullptr; P.unmatched = nullptr; P.pprior = nullptr; P.ntiles = (n_priors + 31) / 32;
  P.index_sum = 0ull;
  P.prior_words = (long long)n_priors * 4 * (prior_dtype == SSDG_F64 ? 8 : 4) / 8;
  if (prior_index) {
    IndexInfo info;
    {
      std::lock_guard<std::mutex> lk(g_index_mu);
      auto it = g_index.find(prior_index);
      if (it == g_index.end()) return SSDG_ERR_ARG;
      info = it->second;
    }
    int dev = 0;
    SSDG_CUDA_TRY(cudaGetDevice(&dev));
    if (info.device != dev) return SSDG_ERR_ARG;
    if (info.n_priors != n_priors || info.dtype != prior_dtype) return SSDG_ERR_SHAPE;
    P.index_sum = info.sum;
    const unsigned char* ib = (const unsigned char*)prior_index;
    P.perm = (const int*)(ib + index_perm_offset());
    P.tiles = (const TileStat*)(ib + index_tiles_offset(n_priors));
    P.supers = (const TileStat*)(ib + index_supers_offset(n_priors));
    P.unmatched = (const float4*)(ib + index_unmatched_offset(n_priors));
    P.pprior = ib + index_pprior_offset(n_priors);
    P.ntiles = info.ntiles;
  }
  SSDG_CUDA_TRY(cudaMemsetAsync(P.ws_head, 0, 256 + align_up((size_t)batch * 4, 256), st));
  P.bits_in_smem = P.elim_words <= kElimSmemWords ? 1 : 0;
  const size_t smem = match_smem_bytes(P.tm, P.ntiles <= kTileSmemMax ? P.ntiles : 0, P.bits_in_smem ? P.elim_words : 0);
  if ((int)smem > max_smem_optin()) return SSDG_ERR_LIMIT;
  if (gt_dtype == SSDG_F32 && prior_dtype == SSDG_F64) return launch_match<float, double>(P, grid, smem, st);
  if (gt_dtype == SSDG_F32 && prior_dtype == SSDG_F32) return launch_match<float, float>(P, grid, smem, st);
  if (gt_dtype == SSDG_F64 && prior_dtype == SSDG_F64) return launch_match<double, double>(P, grid, smem, st);
  return launch_match<double, float>(P, grid, smem, st);
}

extern "C" int ssdg_match_status(const void* workspace, int32_t* status, void* stream) {
  if (!workspace || !status) return SSDG_ERR_ARG;
  u32 head[2];
  SSDG_CUDA_TRY(cudaMemcpyAsync(head, workspace, sizeof(head), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  SSDG_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  *status = (int32_t)head[1];
  return SSDG_OK;
}
