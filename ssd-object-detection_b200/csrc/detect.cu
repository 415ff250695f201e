// Post-processing: softmax score head (models/ssd_model.py:479-488), box decode (:466-467) and the
// per-class score-threshold / top-k / greedy NMS the reference lacks (spec: oracle/ssd_oracle.py
// nms_per_class, IoU formula utils/bbox.py:13-25 in float32).
//
//   filter_kernel  one streaming pass over the logits [B,A,C].  Tiles are 32 priors of ONE image; every CTA owns
//                  one contiguous run of tiles and each of its warps one shared-memory tile at a time, filled
//                  by 1-D bulk TMA (cp.async.bulk + mbarrier).  Row phase, lane r owns row r (stride C words:
//                  conflict-free for odd C): e_c = 2^((x_c - ref) log2e) with the background logit as reference
//                  (one pass; rows that would overflow or lose precision are redone with their maximum), the
//                  sum, one pre-filter bit per class.  Class phase, after a warp transpose of the bit matrices
//                  lane l owns classes l, 32+l, 64+l: exact score e_c * (1/sum) > score_thresh, one shared-memory
//                  atomic per lane and class word reserves slots, and the candidates go STRAIGHT into the
//                  per-(image, class) lists the NMS reads (laid out in prior space, so the CTA's slots cannot
//                  collide with another CTA's): no bucketing pass, no global atomics, nothing to zero.
//                  Optionally leaves per-prior (ref, log sum) and the background CE for the loss, the
//                  probabilities, and the reference's score head.
//   nms_kernel     one CTA per (image, class): exact top-k by (score desc, prior asc) -- radix select when the
//                  list is longer than the sort width, then a bucketed rank sort; the lower-triangle
//                  suppression bits from an interval join (cumulative slab bitsets per axis + width / height
//                  class neighbourhoods, cheap float test with a margin, the exact IEEE formula for the
//                  survivors); rows without suppressors are kept at once, the rest resolved by one warp
//                  iterating "kept(i) <=> no kept j < i suppresses i" to its fixed point.
#include <math_constants.h>
#include <algorithm>
#include <cstring>
#include <type_traits>
#include "common.cuh"

namespace ssdg {

// Filter CTAs: 20 warps = 20 tiles of 32 priors in flight per SM (all the shared memory there is for C = 81) at no more
// than 64 registers per thread, which leaves a third of the register file to the matcher's search CTAs that run
// beside the pass.  Measured (B200, SSD300 B=256): 16 warps 0.163 ms, 20 warps 0.152 ms (0.83 of the copy peak) and
// the chained step 0.520 -> 0.513 ms; without the register cap (96 registers) the pass is as fast but the step is not.
constexpr int kFThreads = 640;
constexpr int kFilterMaxRegs = 64;
constexpr int kFWarps = kFThreads / 32;
// L2 prefetch distance of a filter warp, in tiles.  Measured (B200, SSD300 B=256, filter pass / chained step):
// none 0.1603 / 0.5455 ms, 1 tile 0.1542 / 0.5451 ms (0.82 of the copy peak), 2 tiles 0.1614 / 0.5492 ms,
// 3 tiles 0.1828 / 0.5598 ms; the pass gets slower with every tile beyond the first.
constexpr int kFilterPrefetch = 1;
// Classes between two updates of the filter's pre-filter bound.
constexpr int kFilterPreStep = 16;
constexpr int kNmsThreads = 128;
constexpr int kNmsWarps = kNmsThreads / 32;
constexpr int kSlabs = 32;   // slabs per axis of the NMS candidate join
constexpr int kSizeCls = 16; // width / height classes of the join
constexpr int kABitsD = 21;     // limit on the prior count of a detection call (A < 2^21)

struct DetectParams {
  const float* pred_cls;   // logits (filter) or probabilities (kProbs)
  const float* pred_box;
  const void* priors;
  int B, A, C, tpi;        // tpi: tiles per image
  int tma_ok;              // every tile start / size is 16-byte aligned
  float score_thresh;
  // Candidate lists, one per (image, class), laid out in PRIOR space: [B][C-1][tpi*32] entries
  // (score key << 32) | ~prior.  Every filter CTA owns one contiguous run of `chunk` tiles; inside the list of
  // (image b, class c) it appends to the slots of its own tiles of b -- [32 * first tile, ...) -- through a
  // shared-memory counter, and leaves the count in run_cnt[image][slot][class], slot = CTA - first CTA of the image.
  // No global atomics, no zeroing, no bucketing pass: the NMS reads the one or two (max_slots) runs of its list.
  u64* lists;
  u32* run_cnt;            // [B][max_slots][C-1]
  int chunk, max_li;       // tiles per CTA; images a run can touch (chunk / tpi + 2)
  int max_slots;           // runs an image can be split into (tpi / chunk + 2)
  size_t list_cap;         // tpi*32
  float* boxes;            // [B*A,4] decoded
  float* probs;            // optional [B*A,C]
  float head_thresh;
  float* head_score;
  int* head_cls;
  uint8_t* head_mask;
  float2* row_ml;          // optional [B*A] (row max, log sum exp(x - max)): what the loss needs of this pass
  float* row_negbg;        // optional [B*A] background CE  log-sum - (x_bg - max)   (models/ssd_model.py:362-367)
};

__device__ __forceinline__ u64 evict_first_policy() {
  u64 pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void tma_load_hint(void* smem_dst, const void* gsrc, u32 bytes, u64* bar, u64 pol) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(smem_dst)),
      "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
      : "memory");
}

// models/ssd_model.py:466-467 with scale 1: the reference evaluates np.exp on its float32 offsets, the
// products with the (float64) priors in float64, and stores float32.
template <typename TP>
__device__ __forceinline__ float4 decode_row(float4 t, const void* priors, int a) {
  double dx, dy, dw, dh;
  if (sizeof(TP) == 8) {
    const double2* p = reinterpret_cast<const double2*>(priors) + 2 * (size_t)a;
    double2 u = __ldg(p), v = __ldg(p + 1);
    dx = u.x; dy = u.y; dw = v.x; dh = v.y;
  } else {
    float4 v = __ldg(reinterpret_cast<const float4*>(priors) + a);
    dx = v.x; dy = v.y; dw = v.z; dh = v.w;
  }
  float4 o;
  o.x = (float)((double)t.x * dw + dx);
  o.y = (float)((double)t.y * dh + dy);
  o.z = (float)((double)expf(t.z) * dw);
  o.w = (float)((double)expf(t.w) * dh);
  return o;
}

// 32x32 bit matrix across the warp: lane r passes row r, lane c receives column c (bit r = bit c of row r).
__device__ __forceinline__ u32 warp_transpose32(u32 x, int lane) {
#pragma unroll
  for (int j = 16; j >= 1; j >>= 1) {
    const u32 mk = j == 16 ? 0x0000ffffu : j == 8 ? 0x00ff00ffu : j == 4 ? 0x0f0f0f0fu : j == 2 ? 0x33333333u : 0x55555555u;
    const u32 y = __shfl_xor_sync(SSDG_FULL, x, j);
    x = (lane & j) ? ((x & ~mk) | ((y >> j) & mk)) : ((x & mk) | ((y << j) & ~mk));
  }
  return x;
}

// One warp tile: `rows` priors of image b starting at prior 32*j.
//   row phase    lane r owns row r: max, then  e_c = 2^(x_c*log2e - max*log2e)  (one FFMA + MUFU per class; the
//                rounded constant is the same for every class of the row and cancels in e/sum), the sum, and one
//                pre-filter bit per class (e_c > thresh can only be necessary: the sum is >= ~1).
//   class phase  the bit matrix is transposed, lane l now owns classes l, 32+l, 64+l of ALL rows: candidates
//                cluster in a few rows (weak background) but spread evenly over classes, so the exact test
//                p_c = e_c * (1/sum) > thresh  and the append loop run with balanced lanes.
// kWrite: the rows hold e_c afterwards (probabilities output / score head need them); otherwise e_c is
// recomputed for the few pre-filtered classes.  kProbs: the rows already hold probabilities.
template <typename TP, bool kProbs, bool kWrite>
__device__ __forceinline__ void filter_tile(const DetectParams& P, int b, int j, int rows, float* tile, float2* aux,
                                            int lane, u32* cc, u32 run_off) {   // cc: the CTA's class counters of image b
  const int C = P.C, nfg = P.C - 1;
  const bool valid = lane < rows;
  const int a = j * 32 + lane;
  const long long n = (long long)b * P.A + a;
  float* row = tile + (size_t)(valid ? lane : 0) * C;
  const float thr = P.score_thresh;
  float4 tbox = make_float4(0.f, 0.f, 0.f, 0.f);
  if (!kProbs && valid && P.boxes) tbox = __ldg(reinterpret_cast<const float4*>(P.pred_box) + n);  // early: hide latency
  float inv_s = 1.f, kexp = 0.f;
  // first 96 classes as bit words in registers; more classes fall back to re-testing every class
  float pre = kProbs ? thr : thr * 0.999f;
  u32 bits0 = 0u, bits1 = 0u, bits2 = 0u;
  if (valid) {
    if (!kProbs) {
      // The exponent reference of the row: the true maximum (two passes over the row), or -- when the rows
      // are not overwritten -- first the background logit, which IS the maximum of nearly every trained row:
      // e_c = 2^((x_c - ref) log2e), the common factor cancels in e/sum and in  log sum - (x - ref).  A row
      // whose sum leaves [~1, 2^16] that way (a foreground logit > 11 above the background, NaN, inf) is
      // redone with its maximum, so no input can overflow or lose precision.
      auto row_max = [&]() {
        float m0 = -CUDART_INF_F, m1 = m0, m2 = m0, m3 = m0;
        int c = 0;
        for (; c + 4 <= C; c += 4) {
          m0 = fmaxf(m0, row[c]); m1 = fmaxf(m1, row[c + 1]); m2 = fmaxf(m2, row[c + 2]); m3 = fmaxf(m3, row[c + 3]);
        }
        for (; c < C; ++c) m0 = fmaxf(m0, row[c]);
        return fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
      };
      const float xbg = row[C - 1];
      const bool two_pass = kWrite || nfg > 96;   // rows (or the classes beyond the bit words) are overwritten
      float ref = two_pass ? row_max() : xbg;
      float s0, s1;
      for (int attempt = two_pass ? 1 : 0;; ++attempt) {
        kexp = -ref * SSDG_LOG2E;
        s0 = 0.f; s1 = 0.f;
        auto chunkN = [&](int c0, auto width) {   // `width` classes, fully unrolled: the bit positions are immediates
          constexpr int kW = decltype(width)::value;
          u32 bits = 0u;
          float* r = row + c0;
#pragma unroll
          for (int cc = 0; cc < kW; cc += 2) {
            const float e0 = exp2_ftz(fmaf(r[cc], SSDG_LOG2E, kexp)), e1 = exp2_ftz(fmaf(r[cc + 1], SSDG_LOG2E, kexp));
            if (kWrite) { r[cc] = e0; r[cc + 1] = e1; }
            s0 += e0; s1 += e1;
            if (e0 > pre) bits |= 1u << cc;
            if (e1 > pre) bits |= 2u << cc;
          }
          return bits;
        };
        auto chunk = [&](int c0, int cn) {
          u32 bits = 0u;
          int cc = 0;
          if (cn >= 16) { bits = chunkN(c0, std::integral_constant<int, 16>()); cc = 16; }
          for (; cc < cn; ++cc) {
            const float e0 = exp2_ftz(fmaf(row[c0 + cc], SSDG_LOG2E, kexp));
            if (kWrite) row[c0 + cc] = e0;
            s0 += e0;
            if (e0 > pre) bits |= 1u << cc;
          }
          return bits;
        };
        // p_c > thr needs e_c > thr * sum, and the sum is at least what has been added so far: the pre-filter of
        // the later words tightens with the partial sum, which leaves fewer holes for the class phase
        const float pre0 = pre;
        if (nfg <= 96) {   // the background first: it opens the partial sum (e = 1 when it is the reference)
          const float eb = exp2_ftz(fmaf(xbg, SSDG_LOG2E, kexp));
          if (two_pass) row[C - 1] = eb;
          s0 = eb;
        }
        constexpr int kPs = kFilterPreStep;
        auto word32 = [&](int c0) {
          u32 bits = 0u;
#pragma unroll
          for (int o = 0; o < 32; o += kPs) {
            bits |= chunkN(c0 + o, std::integral_constant<int, kPs>()) << o;
            pre = fmaxf(pre0, pre0 * (s0 + s1));
          }
          return bits;
        };
        auto tail = [&](int c0, int cn) {
          const u32 bits = chunk(c0, cn);
          pre = fmaxf(pre0, pre0 * (s0 + s1));
          return bits;
        };
        bits0 = nfg >= 32 ? word32(0) : tail(0, nfg);
        if (nfg > 32) bits1 = nfg >= 64 ? word32(32) : tail(32, nfg - 32);
        if (nfg > 64) bits2 = nfg >= 96 ? word32(64) : tail(64, nfg - 64);
        pre = pre0;
        for (int c = nfg > 96 ? 96 : C; c < C; ++c) {   // the classes beyond 96 and their background
          const float e0 = exp2_ftz(fmaf(row[c], SSDG_LOG2E, kexp));
          if (two_pass) row[c] = e0;
          s0 += e0;
        }
        if (attempt > 0 || (s0 + s1) <= 65536.f) break;
        ref = row_max();
      }
      inv_s = __frcp_rn(s0 + s1);
      if (P.row_ml) {   // the loss of the same predictions reuses this pass instead of streaming the logits again
        // every e_c carries the common factor 2^d, d = ref*log2e + kexp (the rounding of kexp; exact in one FMA):
        // it cancels in e/sum, the logarithm takes it out explicitly
        const float d = fmaf(ref, SSDG_LOG2E, kexp);
        const float s = s0 + s1;
        const float lg = fmaf(-d, 0.693147180559945f, logf(s));
        P.row_ml[n] = make_float2(ref, lg);
        // With the background as the reference its own term e_bg = 2^d (the same exp2 of the same argument) opens the
        // sum, and the background CE log(s / e_bg) is >= 0: exactly 0 when the rest of the sum is lost in rounding
        // (s == e_bg; the max-shifted formula of the standalone CE pass has log 1 there), else lg, whose rounding of
        // d (either sign, ~1e-7) is held at +0.
        P.row_negbg[n] = xbg != ref ? lg - (xbg - ref) : (s != exp2_ftz(d) && lg > 0.f ? lg : 0.f);
      }
    } else {
      const int lim = min(nfg, 96);
      for (int c = 0; c < lim; ++c) {
        const u32 hit = row[c] > pre ? 1u : 0u;
        if (c < 32) bits0 |= hit << c; else if (c < 64) bits1 |= hit << (c - 32); else bits2 |= hit << (c - 64);
      }
    }
  }
  if (!kProbs) aux[lane] = make_float2(kexp, inv_s);
  // class phase: lane l <-> classes l, 32+l, 64+l; bit r <-> row r
  u32 t0 = warp_transpose32(bits0, lane);                    // includes the __syncwarp the shared writes need
  u32 t1 = nfg > 32 ? warp_transpose32(bits1, lane) : 0u;
  u32 t2 = nfg > 64 ? warp_transpose32(bits2, lane) : 0u;
  __syncwarp();
  auto score_at = [&](float* p, int r) {
    if (kProbs) return *p;
    const float2 ax = aux[r];
    return (kWrite ? *p : exp2_ftz(fmaf(*p, SSDG_LOG2E, ax.x))) * ax.y;
  };
  auto side_outputs = [&]() {   // score head (models/ssd_model.py:481-488) and the decoded box of the lane's row
    if (kProbs || !valid) return;
    if (kWrite && (P.head_score || P.head_cls || P.head_mask)) {
      // max foreground probability, arg-max over all classes (first max)
      float best = row[0];
      int arg = 0;
      float fg = 0.f;
      for (int c = 0; c < C; ++c) {
        const float v = row[c];
        if (v > best) { best = v; arg = c; }
        if (c < C - 1) fg = fmaxf(fg, v);
      }
      const float score = fg * inv_s;
      const float pbg = row[C - 1] * inv_s;
      if (P.head_score) P.head_score[n] = score;
      if (P.head_cls) P.head_cls[n] = arg;
      if (P.head_mask) P.head_mask[n] = (score > P.head_thresh && !(pbg > P.head_thresh)) ? 1 : 0;
    }
    if (P.boxes) reinterpret_cast<float4*>(P.boxes)[n] = decode_row<TP>(tbox, P.priors, a);
  };
  {
    // Straight into the per-(image, class) lists the NMS reads.  The exact test comes first (a pre-filter hit whose
    // score fails leaves nothing; a passing score is parked in the tile element it came from), then ONE shared-memory
    // atomic per lane and class word reserves the lane's slots in the CTA's run of the class list, then the appends.
    // The order inside a run depends on the warps' timing; the NMS sorts by the unique (score, prior) key, so the
    // result does not.
    constexpr bool kStash = !kProbs && !kWrite;   // the tile element is free to hold the score once it has been tested
    auto exact = [&](u32 rb, int c) {   // two hits per trip: the chain load -> exp2 -> compare is latency-bound
      u32 keep = 0u;
      while (rb) {
        const int ra = __ffs(rb) - 1;
        rb &= rb - 1;
        const bool two = rb != 0u;
        const int rb2 = two ? __ffs(rb) - 1 : ra;
        rb &= rb - 1;
        float* pa = tile + ra * C + c;
        float* pb = tile + rb2 * C + c;
        const float sa = score_at(pa, ra), sb = score_at(pb, rb2);
        if (sa > thr) {
          keep |= 1u << ra;
          if (kStash) *pa = sa;
        }
        if (two && sb > thr) {
          keep |= 1u << rb2;
          if (kStash) *pb = sb;
        }
      }
      return keep;
    };
    int c2 = 64 + lane;
    if (nfg > 64 && nfg <= 80) {   // at most 16 classes in the third word: two lanes share a class, 16 rows each
      const u32 lo = __shfl_sync(SSDG_FULL, t2, lane & 15);
      t2 = lane < 16 ? (t2 & 0xffffu) : (lo & 0xffff0000u);
      c2 = 64 + (lane & 15);
    }
    u32 p0 = 0u, p1 = 0u, p2 = 0u;
    const u32 x0 = exact(t0, lane);
    if (x0) p0 = atomicAdd(cc + lane, (u32)__popc(x0));
    const u32 x1 = nfg > 32 ? exact(t1, 32 + lane) : 0u;
    if (x1) p1 = atomicAdd(cc + 32 + lane, (u32)__popc(x1));
    const u32 x2 = nfg > 64 ? exact(t2, c2) : 0u;
    if (x2) p2 = atomicAdd(cc + c2, (u32)__popc(x2));
    u64* lb = P.lists + (size_t)b * nfg * P.list_cap + run_off;
    const u32 nbase = ~(u32)(j * 32);   // ~(32 j + r) = ~(32 j) - r
    auto append = [&](u32 xb, int c, u32 pos) {
      u64* dst = lb + (size_t)c * P.list_cap + pos;
      auto entry = [&](int r) {
        float* p = tile + r * C + c;
        const float score = kStash ? *p : score_at(p, r);
        const u32 sk = kProbs ? key32(score) : (__float_as_uint(score) | 0x80000000u);   // softmax scores are >= +0
        return ((u64)sk << 32) | (u64)(nbase - (u32)r);
      };
      while (xb) {
        const int ra = __ffs(xb) - 1;
        xb &= xb - 1;
        const bool two = xb != 0u;
        const int rb2 = two ? __ffs(xb) - 1 : ra;
        xb &= xb - 1;
        const u64 ea = entry(ra), eb = entry(rb2);
        dst[0] = ea;
        if (two) dst[1] = eb;
        dst += 2;
      }
    };
    append(x0, lane, p0); append(x1, 32 + lane, p1); append(x2, c2, p2);
    if (valid)
      for (int c = 96; c < nfg; ++c) {   // classes beyond the bit words: one atomic per candidate
        const float score = kProbs ? row[c] : row[c] * inv_s;
        if (score > thr) lb[(size_t)c * P.list_cap + atomicAdd(cc + c, 1u)] = ((u64)key32(score) << 32) | (u64)(~(u32)a);
      }
    side_outputs();
  }
  if (kProbs || !valid) return;
  if (kWrite && P.probs)
    for (int c = 0; c < C; ++c) row[c] *= inv_s;
}

// L2 prefetch of a contiguous block (no shared memory, no completion to wait for): keeps DRAM requests in flight for
// tiles whose shared-memory buffer is still being computed on.
__device__ __forceinline__ void prefetch_l2_bulk(const void* gsrc, u32 bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gsrc), "r"(bytes) : "memory");
}

template <typename TP, bool kProbs, bool kWrite>
__global__ void __maxnreg__(kFilterMaxRegs) filter_kernel(DetectParams P, int warps_per_cta, int prefetch) {   // <= 64 registers: leaves room for a matcher CTA
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int C = P.C, A = P.A, tpi = P.tpi, nfg = P.C - 1;
  const size_t tile_floats = (size_t)32 * C;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float* bufs = reinterpret_cast<float*>(smem_raw);
  u64* bars = reinterpret_cast<u64*>(smem_raw + (size_t)warps_per_cta * tile_floats * 4);
  float2* aux = reinterpret_cast<float2*>(bars + kFWarps) + 32 * warp;   // per row: -max*log2e, 1/sum
  u32* scnt = reinterpret_cast<u32*>(reinterpret_cast<float2*>(bars + kFWarps) + 32 * kFWarps);   // [max_li][C-1] class counters of the run
  const int ncnt = P.max_li * nfg;
  for (int i = tid; i < ncnt; i += kFThreads) scnt[i] = 0u;
  if (tid == 0) {
    for (int i = 0; i < warps_per_cta; ++i) mbar_init(&bars[i], 1);
    mbar_fence_init();
  }
  __syncthreads();
  // The CTA's run: tiles [run0, run1) of the batch; the warps interleave inside it.
  const long long run0 = (long long)blockIdx.x * P.chunk;
  const long long run1 = min((long long)P.B * tpi, run0 + P.chunk);
  const int img0 = (int)(run0 / tpi);                 // first image of the run
  const int j0 = (int)(run0 - (long long)img0 * tpi); // its first tile inside that image
  if (warp < warps_per_cta) {
    const long long gw = run0 + warp;
    const int stride = warps_per_cta;
    float* tile = bufs + (size_t)warp * tile_floats;
    u64* mybar = bars + warp;
    const u64 pol = evict_first_policy();

    // (image, tile of the image) of the warp's current tile, advanced without divisions
    int b = (int)(gw / tpi), j = (int)(gw - (long long)b * tpi);
    const int step_b = stride / tpi, step_j = stride - step_b * tpi;
    auto issue = [&](int ib, int ij) {  // lane 0 only
      const u32 bytes = (u32)min(32, A - ij * 32) * (u32)C * 4u;
      mbar_arrive_expect_tx(mybar, bytes);
      tma_load_hint(tile, P.pred_cls + ((size_t)ib * A + (size_t)ij * 32) * C, bytes, mybar, pol);
    };
    // One tile in flight per warp; the other warps of the CTA hide its latency.  That alone leaves too few bytes
    // in flight towards DRAM (a buffer that is being computed on requests nothing): the warp also asks L2 for the
    // tile it will load `prefetch` rounds later, so the bulk copy into shared memory finds its lines in L2.
    // (image, tile) of the tile `prefetch` + 1 rounds ahead, walked like (b, j)
    long long tpf = gw + (long long)(prefetch + 1) * stride;
    int pb = (int)(tpf / tpi), pj = (int)(tpf - (long long)pb * tpi);
    auto prefetch_at = [&](int ib, int ij) {  // lane 0 only
      prefetch_l2_bulk(P.pred_cls + ((size_t)ib * A + (size_t)ij * 32) * C, (u32)min(32, A - ij * 32) * (u32)C * 4u);
    };
    if (P.tma_ok && lane == 0 && gw < run1) {
      issue(b, j);
      for (int d = 1; d <= prefetch; ++d) {
        const long long tp = gw + (long long)d * stride;
        if (tp < run1) prefetch_at((int)(tp / tpi), (int)(tp % tpi));
      }
    }
    int k = 0;
    for (long long t = gw; t < run1; t += stride, ++k) {
      const int rows = min(32, A - j * 32);
      if (P.tma_ok) {
        mbar_wait(mybar, (u32)(k & 1));
      } else {  // unaligned shapes: plain cooperative copy
        const float* g = P.pred_cls + ((size_t)b * A + (size_t)j * 32) * C;
        for (int i = lane; i < rows * C; i += 32) tile[i] = g[i];
        __syncwarp();
      }
      // the run's slots in the lists of image b start at its first tile of b
      filter_tile<TP, kProbs, kWrite>(P, b, j, rows, tile, aux, lane, scnt + (b - img0) * nfg, b == img0 ? (u32)j0 * 32u : 0u);
      // the next bulk copy (async proxy) overwrites rows this warp has just written
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (!kProbs && kWrite && P.probs) {  // the tile layout in shared memory equals the layout in global memory
        float* dst = P.probs + ((size_t)b * A + (size_t)j * 32) * C;
        for (int i = lane; i < rows * C; i += 32) __stcs(&dst[i], tile[i]);
        __syncwarp();
      }
      b += step_b; j += step_j;
      if (j >= tpi) { j -= tpi; ++b; }
      if (P.tma_ok && lane == 0 && t + stride < run1) {
        issue(b, j);
        if (prefetch > 0 && tpf < run1) prefetch_at(pb, pj);
      }
      tpf += stride;
      pb += step_b; pj += step_j;
      if (pj >= tpi) { pj -= tpi; ++pb; }
    }
  }
  __syncthreads();
  // the counts of the run, per image it touched
  const int img1 = run1 > run0 ? (int)((run1 - 1) / tpi) : img0 - 1;
  for (int li = 0; li <= img1 - img0; ++li) {
    const int bi = img0 + li;
    const int slot = (int)blockIdx.x - (int)(((long long)bi * tpi) / P.chunk);
    u32* out = P.run_cnt + ((size_t)bi * P.max_slots + slot) * nfg;
    for (int i = tid; i < nfg; i += kFThreads) out[i] = scnt[li * nfg + i];
  }
}

// ---- per-(image, class) NMS ---------------------------------------------------------------------------
struct NmsParams {
  const u64* lists;    // [B][C-1][list_cap], see DetectParams
  const u32* run_cnt;  // [B][max_slots][C-1]
  size_t list_cap;
  int tpi, chunk, max_slots;
  const float* boxes;  // [B,A,4]
  int A, n_fg, top_k, sortn;  // sortn: power of two >= max(top_k, 32)
  float iou_thresh;
  int* out_kept;
  int* out_count;
  float* out_score;
  // host-computed constants of the join (nms_kernel)
  int B;
  int fast_ok;         // 0 < iou_thresh < 1e6: the division-free pre-test exists
  float q, tq0, inv_l; // thr/(1+thr); shrink factor of the slab intervals; 1 / log2 of the size-class ratio
  u32 key_base;        // score word of the filter's threshold: every listed key's score word lies above it
  float key_scale;     // 256 / (score word of 1.0 - key_base): rank-sort buckets over the scores (thresh, 1]
};

// The NMS kernel is instruction-cache sensitive (12 CTAs per SM in different phases): its block-stride loops
// stay rolled (3280 -> 2240 SASS instructions, 7% faster).
#define NMS_LOOP _Pragma("unroll 1")

// Phase attribution (build with SSDG_EXTRA_NVCC_FLAGS=-DSSDG_NMS_TIMING; profiles/nms_phase_timing.py): thread 0 of
// every CTA reads clock64 after the barrier that ends each phase, the two join passes are clocked per warp, and the
// counts each phase scales with are summed in shared memory; one flush per CTA into g_nms_timing, read (and zeroed)
// by ssdg_nms_timing.  The default build contains none of it.
enum NmsTiming {
  NT_LOAD, NT_SELECT, NT_SCATTER, NT_RANK, NT_OR, NT_JOIN, NT_RESOLVE, NT_OUTPUT,   // CTA cycles per phase
  NT_PASS_A, NT_PASS_B,                 // warp cycles of the two join passes (summed over the warps)
  NT_LISTS, NT_KEYS, NT_SELECTED, NT_ROWS,   // lists, keys loaded, lists through the select, rows kept for the join
  NT_COUNT_STEPS, NT_COUNT_TRIPS,       // count loop: steps summed over threads; trips of the warps (max over lanes)
  NT_A_WORDS,                           // pass A: column words ANDed (per row group)
  NT_B_PAIRS, NT_B_TRIPS, NT_B_WORDS,   // pass B: candidate pairs; trips of the warps; (row, word)s with candidates
  NT_SUPPRESS, NT_OPEN, NT_ROUNDS,      // suppressing pairs; open rows; resolution rounds
  NT_RANK_COUNT, NT_RANK_BOX,           // rank loop, warp cycles: key + count loop; box wait + preparation + registration
  NT_SLOTS = 32
};
#ifdef SSDG_NMS_TIMING
__device__ unsigned long long g_nms_timing[NT_SLOTS];
#define NMS_TICK(slot) do { if (tid == 0) { const long long n_ = clock64(); atomicAdd(&nt_acc[slot], (unsigned long long)(n_ - nt_t0)); nt_t0 = n_; } } while (0)
#define NMS_COUNT(slot, v) atomicAdd(&nt_acc[slot], (unsigned long long)(v))
#define NMS_TIMING_ONLY(...) __VA_ARGS__
#else
#define NMS_TICK(slot) do { } while (0)
#define NMS_COUNT(slot, v) do { } while (0)
#define NMS_TIMING_ONLY(...)
#endif
// Structure (128 threads per list, ~17.8 KB shared memory, <= 40 registers => 12 CTAs per SM; the kernel is
// issue- and barrier-bound, profiles/r20_*, r25_*):
//   * the list is the concatenation of the runs the filter CTAs left in its slots; the counts of up to four runs
//     are fetched together (one memory latency in front of the keys);
//   * exact top-k: a list longer than the sort width goes through an 8-bit radix select of the composite key; then a
//     BUCKETED RANK SORT -- 256 buckets monotone in the key, fixed over the score words (threshold, 1] so that the
//     key load builds the histogram (no range pass); only when every key lands in one bucket (equal or tightly
//     clustered scores) are the buckets rebuilt over the keys' own [min, max] score word (prior word when every
//     score is equal); rank = keys in higher buckets + larger keys in the own bucket.  Exact for any input
//     (clustered scores only lengthen a count loop).  The thread that places a key at rank r < top_k also prepares
//     box r and registers it in the join tables below, so the box load overlaps the count loop;
//   * suppression bits by an INTERVAL JOIN instead of all pairs.  iou(i, j) > t means inter > q (a_i + a_j),
//     q = t / (1 + t); the y overlap is at most min(h_i, h_j), so the x overlap exceeds q (w_i + w_j): the x
//     extents of i and j, each SHRUNK by q times its width at both ends, still meet (same in y).  Every box gets
//     the interval [a, b] of the 32 slabs per axis its shrunk extents touch -- slabs fixed over [0, 1], the ends
//     clamped (a monotone map: clamping only merges slabs); two intervals meet <=> a_j <= b_i and
//     b_j >= a_i.  Per axis two cumulative bitset tables over the boxes, LE[s] = {j : a_j <= s}, GE[s] = {j : b_j >= s}
//     (each box registered at its two end slabs, then a running OR along the slabs), give the x partners of box i as
//     LE[b_i] & GE[a_i]: two loads per axis whatever the width.  SIZE CLASSES prune further: iou > t needs
//     inter > t' E_i and inter <= w_j h_i, so the widths -- and the heights -- of a pair differ by less than 1/t';
//     with classes of that ratio (log2 of the width against the fixed reference 1, clamped) a pair's classes differ
//     by at most one, and two more tables (class neighbourhoods) join the AND.  Survivors get the branch-free float
//     test inter >= 0.9999 q (a_i + a_j), then the formula itself in IEEE float32 (utils/bbox.py:13-25).
//     The bounds are stated in the formula's areas w*h and carry over to the corner extents W, H of a box whose
//     extents reproduce its area to 0.1 % (exact box).  A box j that does not (inexact) is registered UNSHRUNK and in
//     EVERY size class, and as a row it takes all registered boxes as its size partners.  That stays conservative
//     for any partner i: the size classes no longer prune the pair, and in x the unshrunk extent of j meets i's
//     extent shrunk by tq W_i at both ends (tq <= 0.98 q < 1/2) in at least min(ex - tq W_i, (1 - 2 tq) W_i), ex the
//     x overlap of the two boxes; ex >= inter / H_i > q (a_i + a_j) / H_i >= q a_i / H_i >= 0.999 q W_i for an exact
//     i (a_j > 0 for a registered box), so both terms are positive (same in y).  Two inexact boxes are both unshrunk
//     and meet whenever inter > 0.  Thresholds <= 0 or huge use all pairs with the formula;
//   * the join runs per group of 32 rows in two passes (candidate words as straight-line code when the word count
//     is a template constant, then the pair tests, each lane walking its row's candidates through all its words),
//     the groups dealt to the warps in pairs (last + first, ...): group g costs g + 1 words, so every warp gets the
//     same number of word steps;
//   * rows without a suppressor are kept at once; the others (a handful) are listed and resolved by ONE warp
//     iterating the fixed point of kept(i) <=> no kept j < i suppresses i -- identical to the sequential greedy by
//     induction on i, no CTA-wide barrier per round.  The suppression matrix is the lower triangle only,
//     [group][word][row] (conflict-free);
//   * thresholds, shrink factor, class scale and bucket scale come from the host; the slab scale is a constant
//     (any positive scale keeps those maps monotone, which is all the join and the sort need).
template <int kW>   // kW: words of 32 rows (top_k rounded up / 32) as a constant, 0 = any
__global__ void __launch_bounds__(kNmsThreads, 12) nms_kernel(NmsParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int sortn = P.sortn, mcap = (P.top_k + 31) & ~31, W = mcap >> 5, RL = (4 * W) | 1;
  const int RS = (2 * W) | 1;
  const int tabn = (kSlabs * RL + kSizeCls * RS + 3) & ~3;   // words, whole uint4s
  const int supn = 16 * W * (W + 1);
  // Layout: nms_smem_bytes.  The sort scratch (tmp, hist, bstart) and the join's triangle (sup, unres) share one
  // region: the rank loop fills crn / area / qlo / slidx and the tables while it still reads the sort scratch.
  u64* keys = reinterpret_cast<u64*>(smem_raw);                 // [sortn]
  float4* crn = reinterpret_cast<float4*>(keys + sortn);        // [mcap] x1,y1,x2,y2
  u32* tab = reinterpret_cast<u32*>(crn + mcap);                // [kSlabs][RL] interval tables of the join
  u32* stab = tab + kSlabs * RL;                                // [kSizeCls][RS] width / height class neighbourhoods
  float* qlo = reinterpret_cast<float*>(tab + tabn);            // [mcap] q*area*0.9999
  float* area = qlo + mcap;                                     // [mcap]
  u32* slidx = reinterpret_cast<u32*>(area + mcap);             // [mcap] slab intervals and size classes of the box
  u64* tmp = reinterpret_cast<u64*>(slidx + mcap);              // [sortn] rank sort: keys grouped by bucket
  u32* hist = reinterpret_cast<u32*>(tmp + sortn);              // [256] sort / select histogram
  u32* bstart = hist + 256;                                     // [256] rank sort: first slot of each bucket
  u32* sup = slidx + mcap;                                      // lower triangle, [group g][word w <= g][row of the group]
  u32* unres = sup + supn;                                      // [mcap] the open rows, listed
  u32* keptw = slidx + mcap + max(2 * sortn + 512, supn + mcap);   // [W]
  u32* remw = keptw + W;                                        // [W]
  u32* openw = remw + W;                                        // [W] rows with at least one suppressor
  u32* wpre = openw + W;                                        // [W + 1] kept boxes before word w
  __shared__ u64 sel_prefix;
  __shared__ int sel_k, sel_fill;

  const int b = (int)(blockIdx.z * 65535u + blockIdx.y);        // grid (class, image mod 65535, image / 65535)
  if (b >= P.B) return;
#ifdef SSDG_NMS_TIMING
  __shared__ unsigned long long nt_acc[NT_SLOTS];
  long long nt_t0 = clock64();
  if (tid < NT_SLOTS) nt_acc[tid] = 0ull;
#endif
  const size_t list = (size_t)b * P.n_fg + blockIdx.x;
  // The list is the concatenation of the runs the filter CTAs left in its slots (prior space, DetectParams).
  // f(key, index in the list) for every key, block-strided; returns the length.  Everything is derived inside (the
  // counts of the runs fetched together: one memory latency in front of the keys, not one per run), so nothing
  // stays in registers for the rare second use (radix select of an over-long list).
  auto for_keys = [&](auto&& f) -> int {
    const u32 t_lo = (u32)b * (u32)P.tpi;                 // first tile of the image in the batch (tiles < 2^31)
    const u32 s_first = t_lo / (u32)P.chunk;
    const int nruns = (int)((t_lo + (u32)P.tpi - 1u) / (u32)P.chunk - s_first) + 1;
    const u32* rc = P.run_cnt + (size_t)b * P.max_slots * P.n_fg + blockIdx.x;
    const u64* lbase = P.lists + list * P.list_cap;
    // (every thread fetches the counts of the first four runs -- nearly always there are one or two)
    const int c0 = (int)rc[0], c1 = nruns > 1 ? (int)rc[P.n_fg] : 0, c2 = nruns > 2 ? (int)rc[2 * (size_t)P.n_fg] : 0,
              c3 = nruns > 3 ? (int)rc[3 * (size_t)P.n_fg] : 0;
    const u32 chunk32 = (u32)P.chunk * 32u;
    const u32 off1 = ((s_first + 1u) * (u32)P.chunk - t_lo) * 32u;   // slots of the second run (if any)
    int base = 0, mine = 0;
#pragma unroll 1
    for (int r = 0; r < nruns; ++r) {
      int cnt;
      if (r < 4) {
        cnt = r == 0 ? c0 : r == 1 ? c1 : r == 2 ? c2 : c3;
      } else {   // few images on many SMs: 32 more counts per round trip, one per lane
        if (((r - 4) & 31) == 0) mine = r + lane < nruns ? (int)rc[(size_t)(r + lane) * P.n_fg] : 0;
        cnt = __shfl_sync(SSDG_FULL, mine, (r - 4) & 31);
      }
      const u64* ptr = lbase + (r ? off1 + (size_t)(r - 1) * chunk32 : 0);
      NMS_LOOP
      for (int i = tid; i < cnt; i += kNmsThreads) f(ptr[i], base + i);
      base += cnt;
    }
    return base;
  };

  // Sort histogram and join tables start at zero (neither shares memory with anything the key load writes).
  NMS_LOOP
  for (int i = tid; i < (tabn >> 2) + 64; i += kNmsThreads)
    reinterpret_cast<uint4*>(i < (tabn >> 2) ? tab : hist - tabn)[i] = make_uint4(0u, 0u, 0u, 0u);
  if (tid < W) { remw[tid] = 0u; openw[tid] = 0u; }
  __syncthreads();
  // Rank-sort buckets (head of the kernel): first fixed over the score words above the threshold's.
  bool byscore = true;
  u32 kbase = P.key_base;
  float kscale = P.key_scale;
  auto bucket = [&](u64 v) {   // the clamp, the conversions, the product and the truncation are all monotone
    const u32 x = byscore ? (u32)(v >> 32) : (u32)v;
    return min(255, (int)((float)(max(x, kbase) - kbase) * kscale));
  };
  // Lists up to the sort width (all but pathological ones) go straight into the sort buffer and its histogram; a
  // longer one keeps its first sortn keys there only until the select below refills the buffer.
  int n = for_keys([&](u64 v, int i) {
    if (i < sortn) {
      keys[i] = v;
      atomicAdd(&hist[bucket(v)], 1u);
    }
  });
  const bool selected = n > P.sortn;   // more candidates than the sort takes: radix select first
  __syncthreads();
  NMS_TICK(NT_LOAD);
  if (tid == 0) { NMS_COUNT(NT_LISTS, 1); NMS_COUNT(NT_KEYS, n); NMS_COUNT(NT_SELECTED, selected); }
  if (selected) {
    // Radix select of the top_k-th largest composite key (keys are unique), 8 bits per pass.
    if (tid == 0) { sel_prefix = 0ull; sel_k = P.top_k; sel_fill = 0; }
    for (int shift = 56; shift >= 0; shift -= 8) {
      NMS_LOOP
      for (int i = tid; i < 256; i += kNmsThreads) hist[i] = 0u;
      __syncthreads();
      const u64 pre = sel_prefix;
      const u64 hmask = shift == 56 ? 0ull : (~0ull << (shift + 8));
      for_keys([&](u64 v, int) {
        if ((v & hmask) == pre) atomicAdd(&hist[(u32)(v >> shift) & 255u], 1u);
      });
      __syncthreads();
      if (tid == 0) {
        int k = sel_k, acc = 0, d = 255;
#pragma unroll 1
        for (; d > 0; --d) {
          if (acc + (int)hist[d] >= k) break;
          acc += (int)hist[d];
        }
        sel_k = k - acc;
        sel_prefix = pre | ((u64)d << shift);
      }
      __syncthreads();
    }
    const u64 kth = sel_prefix;
    for_keys([&](u64 v, int) {
      if (v >= kth) {
        const int p = atomicAdd(&sel_fill, 1);
        if (p < sortn) keys[p] = v;
      }
    });
    __syncthreads();
    n = min(sel_fill, sortn);
  }
  // The histogram is rebuilt for the keys the select left, and once more, over the keys' own range, when every key
  // sits in one bucket (all scores equal, or within one bucket's width: the count loop would be quadratic).
  for (bool redo = selected, ranged = false;;) {
    if (redo) {
      NMS_LOOP
      for (int i = tid; i < 256; i += kNmsThreads) hist[i] = 0u;
      __syncthreads();
      NMS_LOOP
      for (int i = tid; i < n; i += kNmsThreads) atomicAdd(&hist[bucket(keys[i])], 1u);
      __syncthreads();
    }
    if (ranged || n < 2 || (int)hist[bucket(keys[0])] < n) break;
    u32 hmin = ~0u, hmax = 0u, lmin = ~0u, lmax = 0u;   // range of the score and prior words of the keys
    NMS_LOOP
    for (int i = tid; i < n; i += kNmsThreads) {
      const u64 v = keys[i];
      hmin = min(hmin, (u32)(v >> 32)); hmax = max(hmax, (u32)(v >> 32));
      lmin = min(lmin, (u32)v); lmax = max(lmax, (u32)v);
    }
    hmin = __reduce_min_sync(SSDG_FULL, hmin); hmax = __reduce_max_sync(SSDG_FULL, hmax);
    lmin = __reduce_min_sync(SSDG_FULL, lmin); lmax = __reduce_max_sync(SSDG_FULL, lmax);
    uint4* mm = reinterpret_cast<uint4*>(bstart);   // [kNmsWarps] per-warp ranges (bstart is filled after this)
    if (lane == 0) mm[warp] = make_uint4(hmin, hmax, lmin, lmax);
    __syncthreads();
#pragma unroll
    for (int w = 0; w < kNmsWarps; ++w) {
      const uint4 pw = mm[w];
      hmin = min(hmin, pw.x); hmax = max(hmax, pw.y); lmin = min(lmin, pw.z); lmax = max(lmax, pw.w);
    }
    byscore = hmax > hmin;
    kbase = byscore ? hmin : lmin;
    kscale = __fdividef(256.f, (float)((byscore ? hmax : lmax) - kbase) + 1.f) * 0.999f;
    redo = ranged = true;
  }
  NMS_TICK(NT_SELECT);
  if (warp == 0) {   // start[b] = number of keys in buckets above b; lane l owns buckets 255-8l .. 248-8l
    u32 c[8], tot = 0u;
#pragma unroll
    for (int r = 0; r < 8; ++r) { c[r] = hist[255 - 8 * lane - r]; tot += c[r]; }
    u32 incl = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const u32 v = __shfl_up_sync(SSDG_FULL, incl, o);
      if (lane >= o) incl += v;
    }
    u32 run = incl - tot;
#pragma unroll
    for (int r = 0; r < 8; ++r) { bstart[255 - 8 * lane - r] = run; hist[255 - 8 * lane - r] = run; run += c[r]; }
  }
  __syncthreads();
  NMS_LOOP
  for (int i = tid; i < n; i += kNmsThreads) {
    const u64 v = keys[i];
    tmp[atomicAdd(&hist[bucket(v)], 1u)] = v;   // hist[b] ends as the end of bucket b
  }
  __syncthreads();
  NMS_TICK(NT_SCATTER);
  const int m = min(n, P.top_k);
  const int mpad = (m + 31) & ~31;
  const int ngroups = mpad >> 5;

  // Rank, then -- for the top_k ranks -- the box and its registration in the join tables (head of the kernel).
  // Corners in the formula's own float32 operations (utils/bbox.py:13-21).  qa = q*(area + 0.5e-10):  iou > thr  <=>
  // inter > qa_i + qa_j  in exact arithmetic (positive denominator); boxes that can never overlap anything (w <= 0,
  // h <= 0, non-finite) get qa = +inf and no registration, so the fast test rejects them exactly like the formula
  // does (their intersection is 0).  Rows m .. mpad are left unprepared: no test uses them.
  const float thr = P.iou_thresh;
  const bool fast_ok = P.fast_ok != 0;
  const float q = P.q;
  NMS_LOOP
  for (int i = tid; i < n; i += kNmsThreads) {
    NMS_TIMING_ONLY(const long long nt_r0 = clock64();)
    const u64 v = tmp[i];
    const float4 bx = __ldg(reinterpret_cast<const float4*>(P.boxes) + (size_t)b * P.A + (int)(~(u32)v));
    const int bk = bucket(v);
    const int s0 = (int)bstart[bk], s1 = (int)hist[bk];
    int r = s0;
#pragma unroll 1
    for (int t = s0; t < s1; ++t) r += tmp[t] > v;
    NMS_TIMING_ONLY({   // (__activemask: the lanes still in the loop, not necessarily converged -- these per-warp
                        // trips, and the rank cycles below, are approximate)
      const u32 am = __activemask(), tr = __reduce_max_sync(am, (u32)(s1 - s0)), st = __reduce_add_sync(am, (u32)(s1 - s0));
      if (lane == __ffs(am) - 1) { NMS_COUNT(NT_COUNT_TRIPS, tr); NMS_COUNT(NT_COUNT_STEPS, st); }
    })
    NMS_TIMING_ONLY(const long long nt_r1 = clock64();)
    if (r >= m) continue;
    keys[r] = v;
    const float hw = __fmul_rn(bx.z, 0.5f), hh = __fmul_rn(bx.w, 0.5f);
    const float4 c = make_float4(__fsub_rn(bx.x, hw), __fsub_rn(bx.y, hh), __fadd_rn(bx.x, hw), __fadd_rn(bx.y, hh));
    const float ar = __fmul_rn(bx.z, bx.w);
    crn[r] = c;
    area[r] = ar;
    float qa = CUDART_INF_F;
    u32 sl = 0u;
    if (bx.z > 0.f && bx.w > 0.f && isfinite(c.x) && isfinite(c.y) && isfinite(c.z) && isfinite(c.w) && isfinite(ar)) {
      qa = q * (ar + 0.5e-10f);
      const float pr = (c.z - c.x) * (c.w - c.y);
      const bool exact = ar >= 0.999f * pr && ar <= 1.001f * pr;   // see the head of the kernel for an inexact box
      const float tq = exact ? P.tq0 : 0.f;
      auto slab = [&](float u) {   // monotone in u (the conversion saturates, NaN -> 0)
        return min(max(__float2int_rd(u * (float)kSlabs), 0), kSlabs - 1);
      };
      auto size_cls = [&](float ext) {   // monotone in ext, clamped (clamping only merges classes)
        return exact ? min(max(__float2int_rd(-__log2f(ext) * P.inv_l), 0), kSizeCls - 1) : kSizeCls - 1;
      };
      const float sx = tq * (c.z - c.x) - 1e-6f * (fabsf(c.x) + fabsf(c.z));
      const float sy = tq * (c.w - c.y) - 1e-6f * (fabsf(c.y) + fabsf(c.w));
      const int ax = slab(c.x + sx), bx_ = max(slab(c.z - sx), ax);
      const int ay = slab(c.y + sy), by = max(slab(c.w - sy), ay);
      const int cw = size_cls(c.z - c.x), ch = size_cls(c.w - c.y);
      sl = (u32)ax | ((u32)bx_ << 5) | ((u32)ay << 10) | ((u32)by << 15) | ((u32)cw << 20) | ((u32)ch << 24) |
           (exact ? 0u : 0x40000000u) | 0x80000000u;
      const u32 bit = 1u << (r & 31);
      const int wi = r >> 5;
      atomicOr(&tab[ax * RL + wi], bit);
      atomicOr(&tab[bx_ * RL + W + wi], bit);
      atomicOr(&tab[ay * RL + 2 * W + wi], bit);
      atomicOr(&tab[by * RL + 3 * W + wi], bit);
#pragma unroll 1
      for (int k = exact ? 0 : kSizeCls - 1; k >= 0; --k) {   // an inexact box goes into every class
        atomicOr(&stab[(cw - k) * RS + wi], bit);
        atomicOr(&stab[(ch - k) * RS + W + wi], bit);
      }
    }
    qlo[r] = qa * 0.9999f;
    slidx[r] = sl;
    NMS_TIMING_ONLY({
      const long long nt_r2 = clock64();
      const u32 am = __activemask();
      const u32 c = __reduce_max_sync(am, (u32)(nt_r1 - nt_r0)), p = __reduce_max_sync(am, (u32)(nt_r2 - nt_r1));
      if (lane == __ffs(am) - 1) { NMS_COUNT(NT_RANK_COUNT, c); NMS_COUNT(NT_RANK_BOX, p); }
    })
  }
  __syncthreads();
  NMS_TICK(NT_RANK);
  if (tid == 0) NMS_COUNT(NT_ROWS, m);

  if (fast_ok) {
    // Slab join + size classes (derivation at the head of the kernel): running ORs along the slabs, class
    // neighbourhoods.
    NMS_LOOP
    for (int col = tid; col < 6 * W; col += kNmsThreads) {
      // (the words of a column are loaded into registers before any is stored: a load after a store to the same
      // column would wait for it, one shared-memory round trip per slab)
      if (col < 4 * W) {
        const bool up = ((col / W) & 1) == 0;   // LE: ascending running OR, GE: descending
        const int step = up ? RL : -RL;
        u32* p = tab + col + (up ? 0 : (kSlabs - 1) * RL);
        u32 acc = 0u;
#pragma unroll 1
        for (int k = 0; k < kSlabs; k += 8, p += 8 * step) {
          u32 v[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) v[e] = p[e * step];
#pragma unroll
          for (int e = 0; e < 8; ++e) { acc |= v[e]; p[e * step] = acc; }
        }
      } else {
        u32* sc = stab + (col - 4 * W);
        u32 prev = 0u, cur = sc[0];
#pragma unroll 1
        for (int k = 0; k < kSizeCls; k += 8) {
          u32 v[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) v[e] = k + e + 1 < kSizeCls ? sc[(k + e + 1) * RS] : 0u;
#pragma unroll
          for (int e = 0; e < 8; ++e) { sc[(k + e) * RS] = prev | cur | v[e]; prev = cur; cur = v[e]; }
        }
      }
    }
    __syncthreads();
    NMS_TICK(NT_OR);
    // The join proper, per group of 32 rows (lane = row), in two passes over the column words w <= g:
    //   A  candidate words = AND of the six table words -- straight-line code when the word count is a template
    //      constant (immediate offsets, no address arithmetic), parked in the row's slots of the triangle;
    //   B  every candidate gets the cheap float test (1e-4 margin), survivors the formula itself -- IEEE float32, no
    //      contraction (utils/bbox.py:13-25); each word is rewritten with the real suppressions.
    // Rows that end without a suppressor stay closed (kept at once); the others are opened for the resolution.
    const u32 ltmask = (1u << lane) - 1u;
    auto join_group = [&](int gi) {
      const int i = (gi << 5) + lane;
      const bool live = i < m;
      const u32 si = live ? slidx[i] : 0u;
      const u32 smask = (u32)((int)si >> 31);                    // insane / padding rows: no candidates
      const u32* lex = tab + ((si >> 5) & 31u) * RL;             // LEx[b_i]
      const u32* gex = tab + (si & 31u) * RL + W;                // GEx[a_i]
      const u32* ley = tab + ((si >> 15) & 31u) * RL + 2 * W;    // LEy[b_i]
      const u32* gey = tab + ((si >> 10) & 31u) * RL + 3 * W;    // GEy[a_i]
      // width / height classes next to the row's; an inexact row (bit 30) takes every size: LEx / LEy again
      const bool inx = (si & 0x40000000u) != 0u;
      const u32* szw = inx ? lex : stab + ((si >> 20) & 15u) * RS;
      const u32* szh = inx ? ley : stab + ((si >> 24) & 15u) * RS + W;
      u32* myrow = sup + 16 * gi * (gi + 1) + lane;              // slot of word w: myrow[32 w]
      NMS_TIMING_ONLY(long long nt_w0 = clock64(); u32 nt_pairs = 0u;)
      u32 wm = 0u;   // the row's words that hold candidates
      if (kW > 0) {
#pragma unroll
        for (int w = 0; w < kW; ++w) {
          if (w <= gi) {
            u32 cand = lex[w] & gex[w] & ley[w] & gey[w] & szw[w] & szh[w] & smask;
            if (w == gi) cand &= ltmask;
            myrow[w << 5] = cand;
            if (cand) wm |= 1u << w;
            NMS_TIMING_ONLY(nt_pairs += __popc(cand);)
          }
        }
      } else {
#pragma unroll 1
        for (int w = 0; w <= gi; ++w) {
          u32 cand = lex[w] & gex[w] & ley[w] & gey[w] & szw[w] & szh[w] & smask;
          if (w == gi) cand &= ltmask;
          myrow[w << 5] = cand;
          if (cand) wm |= 1u << w;
          NMS_TIMING_ONLY(nt_pairs += __popc(cand);)
        }
      }
      NMS_TIMING_ONLY({
        __syncwarp();
        const long long n_ = clock64();
        const u32 tr = __reduce_max_sync(SSDG_FULL, nt_pairs), np = __reduce_add_sync(SSDG_FULL, nt_pairs);
        const u32 nw = __reduce_add_sync(SSDG_FULL, (u32)__popc(wm));
        if (lane == 0) {
          NMS_COUNT(NT_PASS_A, n_ - nt_w0); NMS_COUNT(NT_A_WORDS, gi + 1);
          NMS_COUNT(NT_B_TRIPS, tr); NMS_COUNT(NT_B_PAIRS, np); NMS_COUNT(NT_B_WORDS, nw);
        }
        nt_w0 = n_;
      })
      if (!__any_sync(SSDG_FULL, wm != 0u)) return;
      const float4 bi = live ? crn[i] : make_float4(0.f, 0.f, 0.f, 0.f);
      const float qi_lo = live ? qlo[i] : 0.f;
      const float ai = live ? area[i] : 0.f;
      NMS_TIMING_ONLY(u32 nt_sup = 0u;)
      // Each lane walks the candidates of its own row through all its words, one pair per trip: the warp runs the
      // largest candidate count of its rows, not the sum over the words of each word's largest count, and casts no
      // vote per word.  A word is rewritten with its real suppressions after its last candidate.
      u32 any = 0u, cand = 0u, bits = 0u;
      int w = 0;
#pragma unroll 1
      while (wm | cand) {
        if (cand == 0u) {
          w = __ffs(wm) - 1;
          wm &= wm - 1u;
          cand = myrow[w << 5];
        }
        const int jj = __ffs(cand) - 1;
        cand &= cand - 1u;
        const int j = (w << 5) + jj;
        const float4 bj = crn[j];
        const float lox = fmaxf(bi.x, bj.x), hix = fminf(bi.z, bj.z), loy = fmaxf(bi.y, bj.y), hiy = fminf(bi.w, bj.w);
        const float fx = hix - lox, fy = hiy - loy;
        if (fx > 0.f && fx * fy >= qi_lo + qlo[j]) {
          const float ex = fmaxf(0.f, __fsub_rn(hix, lox));
          const float ey = fmaxf(0.f, __fsub_rn(hiy, loy));
          const float inter = __fmul_rn(ex, ey);
          const float den = __fadd_rn(__fsub_rn(__fadd_rn(area[j], ai), inter), 1e-10f);
          if (__fdiv_rn(inter, den) > thr) bits |= 1u << jj;
        }
        if (cand == 0u) {
          myrow[w << 5] = bits;
          any |= bits;
          NMS_TIMING_ONLY(nt_sup += __popc(bits);)
          bits = 0u;
        }
      }
      const u32 open_rows = __ballot_sync(SSDG_FULL, any != 0u);
      if (lane == 0) openw[gi] = open_rows;
      NMS_TIMING_ONLY({
        nt_sup = __reduce_add_sync(SSDG_FULL, nt_sup);
        if (lane == 0) { NMS_COUNT(NT_PASS_B, clock64() - nt_w0); NMS_COUNT(NT_SUPPRESS, nt_sup); }
      })
    };
    // group g costs g + 1 words: dealt in pairs (last + first, ...) every warp gets the same number of word steps
    for (int k = warp; 2 * k < ngroups; k += kNmsWarps) {
      const int hi = ngroups - 1 - k;
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {   // (one copy of the group code: the kernel is instruction-cache sensitive)
        if (h == 1 && hi == k) break;
        join_group(h == 0 ? hi : k);
      }
    }
  } else {
    // No division-free test for this threshold: all pairs, the formula itself.
    // Task (g, w<=g): lane = row 32g+lane, loop over the 32 columns of group w (uniform shared loads).
    const int ntasks = ngroups * (ngroups + 1) / 2;
    for (int task = warp; task < ntasks; task += kNmsWarps) {
      int g = 0;
      while ((g + 1) * (g + 2) / 2 <= task) ++g;
      const int w = task - g * (g + 1) / 2;
      const int i = (g << 5) + lane;
      const float4 bi = crn[i];
      u32 bits = 0u;
      if (i < m) {
        const int jend = w == g ? lane : 32;
        for (int jj = 0; jj < jend; ++jj) {   // IEEE float32, no contraction (utils/bbox.py:13-25)
          const int j = (w << 5) + jj;
          if (j >= m) break;
          const float4 bj = crn[j];
          const float ex = fmaxf(0.f, __fsub_rn(fminf(bi.z, bj.z), fmaxf(bi.x, bj.x)));
          const float ey = fmaxf(0.f, __fsub_rn(fminf(bi.w, bj.w), fmaxf(bi.y, bj.y)));
          const float inter = __fmul_rn(ex, ey);
          const float den = __fadd_rn(__fsub_rn(__fadd_rn(area[j], area[i]), inter), 1e-10f);
          if (__fdiv_rn(inter, den) > thr) bits |= 1u << jj;
        }
      }
      sup[16 * g * (g + 1) + (w << 5) + lane] = bits;
    }
    NMS_LOOP
    for (int g = tid; g < W; g += kNmsThreads)   // every live row is open
      openw[g] = m >= 32 * (g + 1) ? ~0u : (m > 32 * g ? (1u << (m - 32 * g)) - 1u : 0u);
  }
  __syncthreads();
  NMS_TICK(NT_JOIN);

  // Closed rows are kept at once.  The open ones: fixed point of  kept(i) <=> no kept j < i with sup(i, j);
  // removed(i) <=> some kept j < i with sup(i, j), by one warp (a handful of rows per list: no CTA-wide barrier per
  // round); then wpre[w] = kept boxes before word w for the output.
  if (warp == 0) {
    const u32 ow = lane < W ? openw[lane] : 0u;
    const u32 lm = m >= 32 * (lane + 1) ? ~0u : (m > 32 * lane ? (1u << (m - 32 * lane)) - 1u : 0u);
    if (lane < W) keptw[lane] = lm & ~ow;
    const int oc = __popc(ow);
    int oincl = oc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(SSDG_FULL, oincl, o);
      if (lane >= o) oincl += v;
    }
    const int nu = __shfl_sync(SSDG_FULL, oincl, 31);
    {
      u32 t = ow;
      int p = oincl - oc;
      while (t) {
        unres[p++] = (u32)((lane << 5) + __ffs(t) - 1);
        t &= t - 1;
      }
    }
    __syncwarp();
    if (lane == 0) NMS_COUNT(NT_OPEN, nu);
    for (;;) {
      if (lane == 0) NMS_COUNT(NT_ROUNDS, 1);
      bool unknown = false;
      for (int k = lane; k < nu; k += 32) {
        const int i = (int)unres[k], gi = i >> 5;
        const u32 bit = 1u << (i & 31);
        if ((keptw[gi] | remw[gi]) & bit) continue;
        bool hit_kept = false, all_removed = true;
        const int sbase = 16 * gi * (gi + 1) + (i & 31);
#pragma unroll 1
        for (int w = 0; w <= gi; ++w) {
          const u32 sb = sup[sbase + (w << 5)];
          if (sb & keptw[w]) hit_kept = true;
          if (sb & ~remw[w]) all_removed = false;
        }
        if (hit_kept) atomicOr(&remw[gi], bit);
        else if (all_removed) atomicOr(&keptw[gi], bit);
        else unknown = true;
      }
      __syncwarp();
      if (!__any_sync(SSDG_FULL, unknown)) break;
    }
    const int c = lane < W ? __popc(keptw[lane]) : 0;
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(SSDG_FULL, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane < W) wpre[lane] = (u32)(incl - c);   // W <= 32 (shared memory limits sortn to 1024)
    if (lane == 31) wpre[W] = (u32)incl;
  }
  __syncthreads();
  NMS_TICK(NT_RESOLVE);
  int* ok = P.out_kept + list * (size_t)P.top_k;
  float* os = P.out_score ? P.out_score + list * (size_t)P.top_k : nullptr;
  const int total = (int)wpre[W];
  for (int i = total + tid; i < P.top_k; i += kNmsThreads) {
    ok[i] = -1;
    if (os) os[i] = 0.f;
  }
  NMS_LOOP
  for (int i = tid; i < m; i += kNmsThreads) {
    const u32 kw = keptw[i >> 5], bit = 1u << (i & 31);
    if (kw & bit) {
      const int rank = (int)wpre[i >> 5] + __popc(kw & (bit - 1u));
      ok[rank] = (int)(~(u32)keys[i]);
      if (os) os[rank] = unkey32((u32)(keys[i] >> 32));
    }
  }
  if (tid == 0) P.out_count[list] = total;
#ifdef SSDG_NMS_TIMING
  __syncthreads();
  NMS_TICK(NT_OUTPUT);
  __syncthreads();
  if (tid < NT_SLOTS && nt_acc[tid]) atomicAdd(&g_nms_timing[tid], nt_acc[tid]);
#endif
}

// Launch geometry of the filter pass, a pure function of the shape (both stages and the workspace size derive it).
struct FilterGeom {
  int warps;       // tiles in flight per CTA
  int grid, chunk; // CTAs and tiles per CTA (one contiguous run each)
  int max_li;      // images a run can touch
  int max_slots;   // runs an image can be split into
  size_t cnt_bytes, smem;
};
static bool filter_geom(long long batch, int A, int C, FilterGeom* g) {
  const long long tpi = ((long long)A + 31) / 32, tiles = batch * tpi, nfg = C - 1;
  if (tiles <= 0 || tiles > 0x7fffffffll) return false;
  // shared memory: class counters of the run (a few images' worth), then as many 32-prior tiles as fit
  const size_t cnt_budget = std::max<size_t>(8192, (size_t)3 * nfg * 4);
  // one run per SM; a small batch gets fewer CTAs rather than runs shorter than the tiles a CTA has in flight anyway
  // (16: the NMS then reads an SSD300 image in at most 18 runs instead of 273)
  long long chunk = (tiles + sm_count() - 1) / sm_count();
  if (chunk < 16) chunk = tiles < 16 ? tiles : 16;
  if ((size_t)(chunk / tpi + 2) * nfg * 4 > cnt_budget) chunk = std::max<long long>(1, (long long)(cnt_budget / (4 * nfg)) - 2) * tpi;
  g->chunk = (int)chunk;
  g->grid = (int)((tiles + chunk - 1) / chunk);
  g->max_li = (int)(chunk / tpi + 2);
  g->max_slots = (int)(tpi / chunk + 2);
  g->cnt_bytes = align_up((size_t)g->max_li * nfg * 4, 16);
  const size_t budget = 220 * 1024, fixed = (size_t)kFWarps * 8 + (size_t)kFWarps * 32 * 8 + g->cnt_bytes + 128;
  if (budget <= fixed) return false;
  long long w = (long long)((budget - fixed) / ((size_t)32 * C * 4));
  if (w > kFWarps) w = kFWarps;
  if (w > chunk) w = chunk;
  g->warps = (int)w;
  g->smem = (size_t)g->warps * 32 * C * 4 + fixed;
  return w >= 1;
}
static int next_pow2(int v) {
  int p = 32;
  while (p < v) p <<= 1;
  return p;
}
static size_t nms_smem_bytes(int sortn, int top_k) {   // the layout at the head of nms_kernel
  const int mcap = (top_k + 31) & ~31, W = mcap / 32, RL = (4 * W) | 1;
  const size_t tabn = ((size_t)kSlabs * RL + (size_t)kSizeCls * ((2 * W) | 1) + 3) & ~(size_t)3;
  const size_t sort = (size_t)2 * sortn + 512, join = (size_t)16 * W * (W + 1) + mcap;   // words of the shared region
  return (size_t)sortn * 8 + (size_t)mcap * (16 + 4 + 4 + 4) + tabn * 4 + std::max(sort, join) * 4 +
         (size_t)(4 * W + 1) * 4 + 16 + 128;
}

struct DetectWs {
  u32* run_cnt;
  u64* lists;
  float* boxes;
};
static size_t detect_ws_layout(long long batch, int A, int C, DetectWs* out, unsigned char* base) {
  FilterGeom g;
  if (!filter_geom(batch, A, C, &g)) return 0;
  size_t o = 0;
  const size_t tpi = ((size_t)A + 31) / 32;
  const size_t nfg = (size_t)C - 1;
  if (out) out->run_cnt = (u32*)(base + o);
  o += align_up((size_t)batch * g.max_slots * nfg * 4, 256);
  if (out) out->lists = (u64*)(base + o);
  o += align_up((size_t)batch * nfg * tpi * 32 * 8, 256);
  if (out) out->boxes = (float*)(base + o);
  o += align_up((size_t)batch * A * 16, 256);
  return o;
}

// What the filter pass reads: logits with box offsets and priors (ssdg_detect, ssdg_detect_stage), or probabilities
// with the caller's decoded boxes (ssdg_nms; no priors, no side outputs).
enum class DetectMode { kLogits, kProbs };

static int run_filter(DetectParams& P, DetectMode mode, int prior_dtype, cudaStream_t st) {
  FilterGeom g;
  if (!filter_geom(P.B, P.A, P.C, &g)) return SSDG_ERR_LIMIT;
  P.chunk = g.chunk; P.max_li = g.max_li; P.max_slots = g.max_slots;
  P.tma_ok = (((long long)P.A * P.C) % 4 == 0) && (((uintptr_t)P.pred_cls & 15) == 0);
  prof_begin(SSDG_PROF_FILTER, st);
  // kWrite: the rows must hold exp(x - max) after the pass (probabilities output, score head)
  const bool wr = P.probs || P.head_score || P.head_cls || P.head_mask;
  auto go = [&](auto kern) -> int {
    SSDG_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem));
    kern<<<g.grid, kFThreads, g.smem, st>>>(P, g.warps, kFilterPrefetch);
    return SSDG_OK;
  };
  int rc;
  if (mode == DetectMode::kProbs) rc = go(filter_kernel<float, true, false>);
  else if (prior_dtype == SSDG_F64) rc = wr ? go(filter_kernel<double, false, true>) : go(filter_kernel<double, false, false>);
  else rc = wr ? go(filter_kernel<float, false, true>) : go(filter_kernel<float, false, false>);
  if (rc != SSDG_OK) return rc;
  prof_end(SSDG_PROF_FILTER, st);
  SSDG_LAUNCH_CHECK();
  return SSDG_OK;
}

// key32 of the device code (common.cuh) on the host
static u32 host_key32(float v) {
  if (v != v) return ~0u;
  if (v == 0.0f) v = 0.0f;
  u32 b;
  std::memcpy(&b, &v, 4);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

#ifdef SSDG_NMS_TIMING
// Copies the phase attribution of the nms_kernel launches since the last call (NmsTiming slots) and zeroes it.
extern "C" SSDG_API int ssdg_nms_timing(unsigned long long* out, int32_t n) {
  if (!out || n <= 0 || n > NT_SLOTS) return SSDG_ERR_ARG;
  SSDG_CUDA_TRY(cudaDeviceSynchronize());
  SSDG_CUDA_TRY(cudaMemcpyFromSymbol(out, g_nms_timing, (size_t)n * 8));
  static const unsigned long long zero[NT_SLOTS] = {};
  SSDG_CUDA_TRY(cudaMemcpyToSymbol(g_nms_timing, zero, sizeof(zero)));
  return SSDG_OK;
}
#endif

static int run_nms(const DetectWs& ws, const float* boxes, long long batch, int A, int C, int top_k, float score_thresh,
                   float iou_thresh, int* out_kept, int* out_count, float* out_score, cudaStream_t st) {
  FilterGeom g;
  if (!filter_geom(batch, A, C, &g)) return SSDG_ERR_LIMIT;
  NmsParams Q;
  Q.lists = ws.lists; Q.run_cnt = ws.run_cnt;
  Q.tpi = (A + 31) / 32; Q.list_cap = (size_t)Q.tpi * 32; Q.chunk = g.chunk; Q.max_slots = g.max_slots;
  Q.boxes = boxes; Q.A = A; Q.n_fg = C - 1; Q.top_k = top_k;
  Q.sortn = next_pow2(top_k); Q.iou_thresh = iou_thresh;
  Q.out_kept = out_kept; Q.out_count = out_count; Q.out_score = out_score;
  Q.B = (int)batch;
  Q.fast_ok = (iou_thresh > 0.f && iou_thresh < 1e6f) ? 1 : 0;
  Q.q = Q.fast_ok ? iou_thresh / (1.f + iou_thresh) : 0.f;
  Q.tq0 = fminf(0.98f * Q.q, 0.49f);
  {
    const float tp = 0.99f * iou_thresh / (1.f + 0.001f * iou_thresh);
    Q.inv_l = (Q.fast_ok && tp < 0.98f) ? -1.f / log2f(tp) : 0.f;
  }
  // The filter lists only scores > score_thresh; softmax scores are <= 1 (larger ones share the last bucket).
  Q.key_base = host_key32(score_thresh);
  Q.key_scale = 256.f / (float)std::max<long long>((long long)host_key32(1.f) - (long long)Q.key_base, 256);
  const size_t smem = nms_smem_bytes(Q.sortn, top_k);
  if ((int)smem > max_smem_optin()) return SSDG_ERR_LIMIT;
  auto go = [&](auto kern) -> int {
    if (smem > 48 * 1024)
      SSDG_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SSDG_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    // grid (class, image mod 65535, image / 65535): the lists of an image sit next to each other in the launch order
    const dim3 grid((unsigned)(C - 1), (unsigned)(batch < 65535 ? batch : 65535), (unsigned)((batch + 65534) / 65535));
    prof_begin(SSDG_PROF_NMS, st);
    kern<<<grid, kNmsThreads, smem, st>>>(Q);
    prof_end(SSDG_PROF_NMS, st);
    return SSDG_OK;
  };
  int rc;
  switch ((top_k + 31) / 32) {   // the common list lengths get the join's word loop as straight-line code
    case 1: rc = go(nms_kernel<1>); break;
    case 2: rc = go(nms_kernel<2>); break;
    case 3: rc = go(nms_kernel<3>); break;
    case 4: rc = go(nms_kernel<4>); break;
    case 7: rc = go(nms_kernel<7>); break;
    case 8: rc = go(nms_kernel<8>); break;
    default: rc = go(nms_kernel<0>); break;
  }
  if (rc != SSDG_OK) return rc;
  SSDG_LAUNCH_CHECK();
  return SSDG_OK;
}

// ---- per-image keep_top_k (A12) -----------------------------------------------------------------------
// One CTA per image ranks the candidates of its class lists -- the first min(clamp(count, 0, top_k), K) entries of
// each (nothing beyond can be selected) -- by (score desc, class asc, position asc) and keeps the first K:
//   * the per-class lengths and their prefix in shared memory;
//   * more than K candidates: a radix select (8 bits x 4 passes) finds the K-th largest score key t and how many of
//     the entries equal to t are taken.  When every list's candidate slots fit (kTopkCache keys: SSD300's 80 x 200
//     do), one coalesced pass copies the score keys into shared memory first; otherwise every pass reads them from
//     global memory.  A pass walks each class list with one warp and counts RUNS of equal digits (a run of digit d
//     over [s, e] adds e + 1 - s to bin d): score-sorted lists have a handful of runs, so the shared-memory atomics
//     are few and rarely contended -- and the counts are exact for any order of the entries;
//   * per class, one warp counts the entries > t and == t; the ties go to the classes in ascending order (a prefix
//     over the tie counts), so every class keeps a prefix m_c of its list -- a valid count array itself;
//   * the survivors get the unique key  key32(score) << 32 | (2047 - class) << 10 | (1023 - position)  and a rank
//     sort (rank = number of larger keys, K <= 1024) puts them in place; the outputs are written in rank order.
constexpr int kTopkThreads = 512;
constexpr int kTopkWarps = kTopkThreads / 32;
constexpr int kTopkCache = 16384;   // score keys cached in shared memory (64 KB)

struct TopkParams {
  const int* kept;           // [B][nfg][top_k]
  const int* count;          // [B][nfg]
  const float* score;        // [B][nfg][top_k]
  const float* boxes;        // [B][A][4] or null
  int A, nfg, top_k, K;
  int cache;                 // nfg * min(top_k, K) when that fits kTopkCache (the cache holds [nfg][min(top_k, K)]), else 0
  int* out_prior;            // [B][K]
  int* out_class;            // [B][K]
  float* out_score;          // [B][K]
  float* out_box;            // [B][K][4] or null
  int* out_n;                // [B]
  int* out_count;            // [B][nfg] or null
};

// In-place exclusive scan of a[0, n) in shared memory, a[n] = total; every thread calls it.
__device__ __forceinline__ void topk_block_scan(u32* a, int n, u32* wsum) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int per = (n + kTopkThreads - 1) / kTopkThreads;
  const int lo = min(n, tid * per), hi = min(n, lo + per);
  u32 s = 0u;
  for (int i = lo; i < hi; ++i) s += a[i];
  u32 incl = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const u32 v = __shfl_up_sync(SSDG_FULL, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  u32 run = incl - s + __reduce_add_sync(SSDG_FULL, lane < warp ? wsum[lane] : 0u);   // the warps before this one
  for (int i = lo; i < hi; ++i) {
    const u32 v = a[i];
    a[i] = run;
    run += v;
  }
  if (tid == kTopkThreads - 1) a[n] = run;   // the last thread's range ends the array (later ranges are empty)
  __syncthreads();
}

__global__ void __launch_bounds__(kTopkThreads) keep_top_k_kernel(TopkParams P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int nfg = P.nfg, K = P.K, top_k = P.top_k;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  u64* skey = reinterpret_cast<u64*>(smem_raw);                    // [K] survivor keys
  u32* len = reinterpret_cast<u32*>(skey + K);                     // [nfg] candidates, later survivors, per class
  u32* off = len + nfg;                                            // [nfg + 1] their prefix
  u32* cgt = off + nfg + 1;                                        // [nfg] entries > t per class
  u32* ceq = cgt + nfg;                                            // [nfg + 1] entries == t per class, then their prefix
  u32* hist = ceq + nfg + 1;                                       // [256]
  u32* wsum = hist + 256;                                          // [kTopkWarps]
  u32* cache = wsum + kTopkWarps;                                  // [nfg][lim] score keys (P.cache > 0)
  __shared__ u32 sel_prefix, sel_k;

  const long long b = blockIdx.x;
  const int* cnt = P.count + b * nfg;
  const size_t row0 = (size_t)b * nfg;                              // first list of the image
  const int lim = min(top_k, K);
  for (int c = tid; c < nfg; c += kTopkThreads) {
    off[c] = len[c] = (u32)min(max(cnt[c], 0), lim);
  }
  __syncthreads();
  topk_block_scan(off, nfg, wsum);
  const u32 total = off[nfg];
  u32 n = total;
  const bool cached = P.cache > 0 && total > (u32)K;   // the keys are copied only for a select
  auto key = [&](int c, int j) {
    return cached ? cache[c * lim + j] : key32(P.score[(row0 + c) * top_k + j]);
  };
  if (total > (u32)K) {
    if (cached) {   // eight independent loads in flight per thread; slots past a list's length are never read
      const u32 nslot = (u32)P.cache;
      for (u32 i0 = tid; i0 < nslot; i0 += 8 * kTopkThreads) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const u32 i = i0 + u * kTopkThreads, c = i / (u32)lim, j = i - c * (u32)lim;
          v[u] = (i < nslot && j < len[c]) ? P.score[(row0 + c) * top_k + j] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const u32 i = i0 + u * kTopkThreads;
          if (i < nslot) cache[i] = key32(v[u]);
        }
      }
    }
    if (tid == 0) { sel_prefix = 0u; sel_k = (u32)K; }
    // Radix select of the K-th largest score key (with multiplicity), 8 bits per pass.
#pragma unroll 1
    for (int shift = 24; shift >= 0; shift -= 8) {
      for (int i = tid; i < 256; i += kTopkThreads) hist[i] = 0u;
      __syncthreads();
      const u32 pre = sel_prefix;
      const u32 hmask = shift == 24 ? 0u : (~0u << (shift + 8));
      constexpr u32 kNone = 0xffffffffu;   // an entry outside the prefix (or past the list)
      for (int c = warp; c < nfg; c += kTopkWarps) {
        const int L = (int)len[c];
        u32 prev = kNone;                  // digit of entry j0 - 1
        for (int j0 = 0; j0 < L; j0 += 32) {
          const int j = j0 + lane;
          u32 d = kNone;
          if (j < L) {
            const u32 k = key(c, j);
            if ((k & hmask) == pre) d = (k >> shift) & 255u;
          }
          u32 dp = __shfl_up_sync(SSDG_FULL, d, 1);
          if (lane == 0) dp = prev;
          prev = __shfl_sync(SSDG_FULL, d, min(31, L - 1 - j0));
          if (j < L && d != dp) {          // a run of dp ends at j - 1, a run of d starts at j
            if (dp != kNone) atomicAdd(&hist[dp], (u32)j);
            if (d != kNone) atomicSub(&hist[d], (u32)j);
          }
        }
        if (lane == 0 && prev != kNone) atomicAdd(&hist[prev], (u32)L);   // the last run ends the list
      }
      __syncthreads();
      if (warp == 0) {   // lane l owns digits 255-8l .. 248-8l; the digit where the count from the top reaches sel_k
        u32 h[8], tot = 0u;
#pragma unroll
        for (int r = 0; r < 8; ++r) { h[r] = hist[255 - 8 * lane - r]; tot += h[r]; }
        u32 incl = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const u32 v = __shfl_up_sync(SSDG_FULL, incl, o);
          if (lane >= o) incl += v;
        }
        const u32 kk = sel_k;
        u32 above = incl - tot;
        __syncwarp();
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          if (above < kk && above + h[r] >= kk) {
            sel_prefix = pre | ((u32)(255 - 8 * lane - r) << shift);
            sel_k = kk - above;
          }
          above += h[r];
        }
      }
      __syncthreads();
    }
    const u32 t = sel_prefix, take = sel_k;   // the K-th largest key; how many of the keys == t are kept
    for (int c = warp; c < nfg; c += kTopkWarps) {
      const int L = (int)len[c];
      u32 g = 0u, e = 0u;
      for (int j = lane; j < L; j += 32) {
        const u32 k = key(c, j);
        g += k > t;
        e += k == t;
      }
      g = __reduce_add_sync(SSDG_FULL, g);
      e = __reduce_add_sync(SSDG_FULL, e);
      if (lane == 0) { cgt[c] = g; ceq[c] = e; }
    }
    __syncthreads();
    topk_block_scan(ceq, nfg, wsum);
    for (int c = tid; c < nfg; c += kTopkThreads) {   // the ties go to the classes in ascending order
      const u32 e = ceq[c + 1] - ceq[c];
      const u32 rest = take > ceq[c] ? take - ceq[c] : 0u;
      off[c] = len[c] = cgt[c] + min(e, rest);
    }
    __syncthreads();
    topk_block_scan(off, nfg, wsum);
    n = off[nfg];   // == K: the histograms are exact, so t is the K-th largest key and take <= its multiplicity
  }
  // the survivors: the prefix len[c] of every list, at off[c] in class order
  for (int c = warp; c < nfg; c += kTopkWarps) {
    const int m = (int)len[c];
    for (int j = lane; j < m; j += 32)
      skey[off[c] + j] = ((u64)key(c, j) << 32) | ((u64)(2047 - c) << 10) | (u64)(1023 - j);
  }
  if (P.out_count)
    for (int c = tid; c < nfg; c += kTopkThreads) P.out_count[row0 + c] = (int)len[c];
  __syncthreads();
  // rank sort, descending (the keys are unique): each thread ranks up to K / kTopkThreads keys in one sweep
  constexpr int kPer = 1024 / kTopkThreads;
  u64 v[kPer];
  u32 rank[kPer];
#pragma unroll
  for (int q = 0; q < kPer; ++q) {
    const u32 i = (u32)(tid + q * kTopkThreads);
    v[q] = i < n ? skey[i] : ~0ull;
    rank[q] = 0u;
  }
  for (u32 s = 0; s < n; ++s) {
    const u64 x = skey[s];
#pragma unroll
    for (int q = 0; q < kPer; ++q) rank[q] += x > v[q];
  }
  const size_t o0 = (size_t)b * K;
#pragma unroll
  for (int q = 0; q < kPer; ++q) {
    if ((u32)(tid + q * kTopkThreads) >= n) break;
    const int c = 2047 - (int)((v[q] >> 10) & 2047u), j = 1023 - (int)(v[q] & 1023u);
    const size_t g = (row0 + c) * top_k + j;
    const int p = P.kept[g];
    const size_t o = o0 + rank[q];
    P.out_prior[o] = p;
    P.out_class[o] = c;
    P.out_score[o] = P.score[g];
    if (P.out_box) {   // a prior index outside [0, A) is never dereferenced
      const float4 bx = (p >= 0 && p < P.A) ? __ldg(reinterpret_cast<const float4*>(P.boxes) + (size_t)b * P.A + p)
                                            : make_float4(0.f, 0.f, 0.f, 0.f);
      reinterpret_cast<float4*>(P.out_box)[o] = bx;
    }
  }
  for (u32 r = n + tid; r < (u32)K; r += kTopkThreads) {
    P.out_prior[o0 + r] = -1;
    P.out_class[o0 + r] = -1;
    P.out_score[o0 + r] = 0.f;
    if (P.out_box) reinterpret_cast<float4*>(P.out_box)[o0 + r] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  if (tid == 0) P.out_n[b] = (int)n;
}

static size_t topk_smem_bytes(int nfg, int K, int cache) {
  return (size_t)K * 8 + ((size_t)4 * nfg + 2 + 256 + kTopkWarps + (size_t)cache) * 4;
}

}  // namespace ssdg

using namespace ssdg;

extern "C" size_t ssdg_detect_workspace_bytes(int64_t batch, int32_t n_priors, int32_t n_classes, int32_t top_k) {
  (void)top_k;
  if (batch <= 0 || n_priors <= 0 || n_classes < 2) return 0;
  return detect_ws_layout(batch, n_priors, n_classes, nullptr, nullptr);
}

// Stage bits of detect_run.
constexpr int kDetectFilter = 1;   // softmax filter + decode + the per-(image, class) candidate lists
constexpr int kDetectNms = 2;      // per-class NMS of the lists the filter left in the workspace

// The core of ssdg_detect, ssdg_detect_stage and ssdg_nms.  scores: logits (DetectMode::kLogits, with pred_box, priors
// and the optional side outputs) or probabilities (kProbs: prior_dtype is SSDG_F32 and pred_box, priors, out_probs,
// head_* and the row statistics are NULL, so their checks pass).  boxes: the decoded boxes the NMS reads -- for logits an optional output of the
// filter (NULL: they stay in the workspace), for probabilities the caller's input (only read).
static int detect_run(DetectMode mode, int stages, const float* scores, const float* pred_box, const void* priors,
                      int32_t prior_dtype, int64_t batch, int32_t n_priors, int32_t n_classes, float score_thresh,
                      int32_t top_k, float iou_thresh, int32_t* out_kept, int32_t* out_count, float* out_kept_score,
                      float* boxes, float* out_probs, float head_thresh, float* head_score, int32_t* head_cls,
                      uint8_t* head_mask, float* out_row_ml, float* out_row_negbg, void* workspace,
                      size_t workspace_bytes, void* stream) {
  if ((out_row_ml == nullptr) != (out_row_negbg == nullptr)) return SSDG_ERR_ARG;
  if (((uintptr_t)out_row_ml & 7) || ((uintptr_t)out_row_negbg & 3)) return SSDG_ERR_ALIGN;
  if (!scores || !out_kept || !out_count) return SSDG_ERR_ARG;
  if (mode == DetectMode::kLogits ? (!pred_box || !priors) : !boxes) return SSDG_ERR_ARG;
  if (batch <= 0 || n_priors <= 0 || n_classes < 2 || top_k <= 0) return SSDG_ERR_ARG;
  if (prior_dtype != SSDG_F32 && prior_dtype != SSDG_F64) return SSDG_ERR_ARG;
  if (top_k > 1024 || batch > 0x7fffffff / 64 || n_priors >= (1 << kABitsD) || n_classes > 2048) return SSDG_ERR_LIMIT;
  if (((uintptr_t)pred_box | (uintptr_t)priors | (uintptr_t)boxes) & 15) return SSDG_ERR_ALIGN;
  if (((uintptr_t)scores | (uintptr_t)out_probs) & 3) return SSDG_ERR_ALIGN;
  if (!workspace || ((uintptr_t)workspace & 255) ||
      workspace_bytes < ssdg_detect_workspace_bytes(batch, n_priors, n_classes, top_k))
    return SSDG_ERR_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  DetectWs ws;
  detect_ws_layout(batch, n_priors, n_classes, &ws, (unsigned char*)workspace);
  DetectParams P{};
  P.pred_cls = scores; P.pred_box = pred_box; P.priors = priors;
  P.B = (int)batch; P.A = n_priors; P.C = n_classes; P.tpi = (n_priors + 31) / 32;
  P.score_thresh = score_thresh;
  P.lists = ws.lists; P.run_cnt = ws.run_cnt; P.list_cap = (size_t)P.tpi * 32;
  P.boxes = boxes ? boxes : ws.boxes; P.probs = out_probs;
  P.head_thresh = head_thresh; P.head_score = head_score; P.head_cls = head_cls; P.head_mask = head_mask;
  P.row_ml = reinterpret_cast<float2*>(out_row_ml); P.row_negbg = out_row_negbg;
  if (stages & kDetectFilter) {
    const int rc = run_filter(P, mode, prior_dtype, st);
    if (rc) return rc;
  }
  if (stages & kDetectNms)
    return run_nms(ws, P.boxes, batch, n_priors, n_classes, top_k, score_thresh, iou_thresh, out_kept, out_count,
                   out_kept_score, st);
  return SSDG_OK;
}

extern "C" int ssdg_detect(const float* pred_cls, const float* pred_box, const void* priors, int32_t prior_dtype,
                           int64_t batch, int32_t n_priors, int32_t n_classes, float score_thresh, int32_t top_k,
                           float iou_thresh, int32_t* out_kept, int32_t* out_count, float* out_kept_score,
                           float* out_boxes, float* out_probs, float head_thresh, float* head_score,
                           int32_t* head_cls, uint8_t* head_mask, void* workspace, size_t workspace_bytes,
                           void* stream) {
  return detect_run(DetectMode::kLogits, kDetectFilter | kDetectNms, pred_cls, pred_box, priors, prior_dtype, batch,
                    n_priors, n_classes, score_thresh, top_k, iou_thresh, out_kept, out_count, out_kept_score,
                    out_boxes, out_probs, head_thresh, head_score, head_cls, head_mask, nullptr, nullptr, workspace,
                    workspace_bytes, stream);
}

extern "C" int ssdg_detect_stage(int32_t stage, const float* pred_cls, const float* pred_box, const void* priors,
                                 int32_t prior_dtype, int64_t batch, int32_t n_priors, int32_t n_classes,
                                 float score_thresh, int32_t top_k, float iou_thresh, int32_t* out_kept,
                                 int32_t* out_count, float* out_kept_score, float* out_boxes, float* out_probs,
                                 float head_thresh, float* head_score, int32_t* head_cls, uint8_t* head_mask,
                                 float* out_row_ml, float* out_row_negbg, void* workspace, size_t workspace_bytes,
                                 void* stream) {
  if (stage != 0 && stage != 1) return SSDG_ERR_ARG;
  return detect_run(DetectMode::kLogits, stage == 0 ? kDetectFilter : kDetectNms, pred_cls, pred_box, priors,
                    prior_dtype, batch, n_priors, n_classes, score_thresh, top_k, iou_thresh, out_kept, out_count,
                    out_kept_score, out_boxes, out_probs, head_thresh, head_score, head_cls, head_mask, out_row_ml,
                    out_row_negbg, workspace, workspace_bytes, stream);
}

extern "C" int ssdg_nms(const float* probs, const float* boxes, int64_t batch, int32_t n_priors, int32_t n_classes,
                        float score_thresh, int32_t top_k, float iou_thresh, int32_t* out_kept, int32_t* out_count,
                        float* out_kept_score, void* workspace, size_t workspace_bytes, void* stream) {
  return detect_run(DetectMode::kProbs, kDetectFilter | kDetectNms, probs, nullptr, nullptr, SSDG_F32, batch, n_priors,
                    n_classes, score_thresh, top_k, iou_thresh, out_kept, out_count, out_kept_score,
                    const_cast<float*>(boxes), nullptr, 0.f, nullptr, nullptr, nullptr, nullptr, nullptr, workspace,
                    workspace_bytes, stream);
}

extern "C" int ssdg_detect_keep_top_k(const int32_t* kept, const int32_t* count, const float* kept_score, int32_t top_k,
                                      const float* boxes, int64_t batch, int32_t n_priors, int32_t n_classes,
                                      int32_t keep_top_k, int32_t* out_prior, int32_t* out_class, float* out_score,
                                      float* out_box, int32_t* out_n, int32_t* out_count, void* stream) {
  if (!kept || !count || !kept_score || !out_prior || !out_class || !out_score || !out_n) return SSDG_ERR_ARG;
  if (out_box && (!boxes || n_priors <= 0)) return SSDG_ERR_ARG;
  if (batch <= 0 || top_k <= 0 || n_classes < 2 || keep_top_k <= 0) return SSDG_ERR_ARG;
  if (top_k > 1024 || keep_top_k > 1024 || n_classes > 2048 || batch > 0x7fffffff / 64) return SSDG_ERR_LIMIT;
  if (((uintptr_t)boxes | (uintptr_t)out_box) & 15) return SSDG_ERR_ALIGN;
  TopkParams P;
  P.kept = kept; P.count = count; P.score = kept_score; P.boxes = boxes;
  P.A = n_priors; P.nfg = n_classes - 1; P.top_k = top_k; P.K = keep_top_k;
  // every list's candidate slots in shared memory when they fit kTopkCache keys (else the select reads global memory)
  const long long slots = (long long)P.nfg * std::min(top_k, keep_top_k);
  P.cache = slots <= kTopkCache ? (int)slots : 0;
  P.out_prior = out_prior; P.out_class = out_class; P.out_score = out_score; P.out_box = out_box;
  P.out_n = out_n; P.out_count = out_count;
  const size_t smem = topk_smem_bytes(P.nfg, P.K, P.cache);
  if ((int)smem > max_smem_optin()) return SSDG_ERR_LIMIT;
  if (smem > 48 * 1024)
    SSDG_CUDA_TRY(cudaFuncSetAttribute(keep_top_k_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  keep_top_k_kernel<<<(unsigned)batch, kTopkThreads, smem, (cudaStream_t)stream>>>(P);
  SSDG_LAUNCH_CHECK();
  return SSDG_OK;
}
