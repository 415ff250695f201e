// Multibox loss with batch-global 3:1 hard-negative mining (models/ssd_model.py:341-396).
//
//   ce_kernel      one streaming pass over the logits [N,C] (N = B*A).  Each warp owns a ring of
//                  32-prior tiles filled by 1-D bulk TMA (cp.async.bulk + mbarrier); lane r then
//                  reads row r from shared memory (stride C words: conflict-free for odd C) and
//                  produces  log-sum-exp, the ground-truth CE of positives, the background CE of
//                  non-positives (the mining input, :362-367), the L1 box term (:384-386), and
//                  the top-11-bit histogram of the mining input.
//   select_kernel  x2: radix select of the k-th largest background CE (k = ratio*num_pos, :368-369)
//                  on the order-preserving key, 11 + 11 + 10 bits, over the L2-resident vector.
//   final_kernel   mask = ce >= k-th (:372, ties kept), masked sum / count, pos&neg overlap check
//                  (:375), deterministic reduction of the per-CTA partials, result block.
//   grad_kernel    optional second pass: d total / d logits and d total / d pred_box (:248).
#include <math_constants.h>
#include <cstddef>
#include "common.cuh"

namespace ssdg {

constexpr int kCeThreads = 256;
constexpr int kCeWarps = kCeThreads / 32;
constexpr int kStages = 2;
constexpr int kBins = 2048;

struct LossWs {
  // device-side layout of the workspace head (all 8-byte aligned)
  double part[256][4];      // per-CTA: sum pos CE, sum L1, num_pos, (unused)
  double fpart[1024][2];    // per-CTA of final_kernel: masked sum, (unused)
  u32 fcount[1024][2];      // per-CTA: neg count, pos&neg overlap count
  u32 hist[3][kBins];       // the three radix levels
  u32 ticket[4];            // last-block-done counters
  u32 nparts[4];            // [0] grid size of the CE pass, [1] positives whose class id is outside [0, C)
  unsigned long long xnpos; // number of positives as an integer: the exchange word of the cross-shard mining
  unsigned long long xpad;
};

struct LossParams {
  const int* gt_cls;
  const float* gt_box;
  const uint8_t* gt_mask;
  const float* pred_box;
  const float* pred_cls;
  long long N;
  int C, ratio;
  float* neg_ce;        // [N] mining input
  uint8_t* neg_mask;    // optional
  double* result;       // [SSDG_LOSS_RESULT_LEN]
  LossWs* ws;
  float* grad_box;
  float* grad_cls;
  const float2* row_ml; // optional: per-prior (max, log-sum) left by the filter pass of the same logits
  const float* row_negbg;   // optional: per-prior background CE from the same pass
  long long N_all;      // priors of the whole (cross-shard) batch; == N for single-shard mining
  int global;           // 1: num_pos and the histograms in the workspace are cross-shard sums
};

__device__ __forceinline__ u64 make_evict_first_policy() {
  u64 pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void tma_load_1d_hint(void* smem_dst, const void* gsrc, u32 bytes, u64* bar, u64 pol) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(smem_dst)),
      "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
      : "memory");
}

// Row statistics from a shared-memory row: max, sum exp(x - max).  Four independent chains.
__device__ __forceinline__ void row_lse(const float* __restrict__ row, int C, float& m, float& s) {
  float m0 = -CUDART_INF_F, m1 = m0, m2 = m0, m3 = m0;
  int c = 0;
  for (; c + 4 <= C; c += 4) {
    m0 = fmaxf(m0, row[c]); m1 = fmaxf(m1, row[c + 1]); m2 = fmaxf(m2, row[c + 2]); m3 = fmaxf(m3, row[c + 3]);
  }
  for (; c < C; ++c) m0 = fmaxf(m0, row[c]);
  m = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  const float nml = m;
  c = 0;
  for (; c + 4 <= C; c += 4) {
    s0 += exp_shifted(row[c], nml); s1 += exp_shifted(row[c + 1], nml);
    s2 += exp_shifted(row[c + 2], nml); s3 += exp_shifted(row[c + 3], nml);
  }
  for (; c < C; ++c) s0 += exp_shifted(row[c], nml);
  s = (s0 + s1) + (s2 + s3);
}

struct CeAcc {
  float pos_ce, l1;
  int npos;
};

// Positive prior n adds ce_of(its ground-truth class), its L1 box distance and 1 to the thread's sums.
template <typename CeOf>
__device__ __forceinline__ void add_positive(const LossParams& P, long long n, CeOf ce_of, CeAcc& acc) {
  int lab = P.gt_cls[n];
  if (lab < 0 || lab >= P.C) {   // TensorFlow raises here (models/ssd_model.py:357): flagged through the status word
    atomicAdd(&P.ws->nparts[1], 1u);
    lab = lab < 0 ? 0 : P.C - 1;
  }
  acc.pos_ce += ce_of(lab);
  const float4 pb = __ldg(reinterpret_cast<const float4*>(P.pred_box) + n);
  const float4 gb = __ldg(reinterpret_cast<const float4*>(P.gt_box) + n);
  acc.l1 += (fabsf(pb.x - gb.x) + fabsf(pb.y - gb.y)) + (fabsf(pb.z - gb.z) + fabsf(pb.w - gb.w));
  acc.npos += 1;
}

// The end of a CE pass (kCeThreads threads): the CTA's three sums in double, reduced in a fixed order into
// ws->part[blockIdx.x]; the grid size, the integer positives count and the CTA's level-0 histogram.
__device__ __forceinline__ void ce_pass_flush(const LossParams& P, const CeAcc& acc, const u32* hist,
                                              double* red /*[3][kCeWarps]*/, int tid) {
  const int lane = tid & 31, warp = tid >> 5;
  double a = warp_sum((double)acc.pos_ce), b = warp_sum((double)acc.l1), c = warp_sum((double)acc.npos);
  if (lane == 0) { red[warp] = a; red[kCeWarps + warp] = b; red[2 * kCeWarps + warp] = c; }
  __syncthreads();
  if (tid == 0) {
    double sa = 0, sb = 0, sc = 0;
    for (int w = 0; w < kCeWarps; ++w) { sa += red[w]; sb += red[kCeWarps + w]; sc += red[2 * kCeWarps + w]; }
    P.ws->part[blockIdx.x][0] = sa; P.ws->part[blockIdx.x][1] = sb; P.ws->part[blockIdx.x][2] = sc;
    if (blockIdx.x == 0) P.ws->nparts[0] = gridDim.x;
    atomicAdd(&P.ws->xnpos, (unsigned long long)sc);   // integer, order-independent
  }
  for (int i = tid; i < kBins; i += kCeThreads) {
    const u32 v = hist[i];
    if (v) atomicAdd(&P.ws->hist[0][i], v);
  }
}

// Per-prior work shared by the TMA path and the tail path.
__device__ __forceinline__ void ce_one_prior(const LossParams& P, long long n, const float* row, u32* hist, CeAcc& acc) {
  const int C = P.C;
  float m, s;
  row_lse(row, C, m, s);
  const float lg = logf(s);
  const bool pos = P.gt_mask[n] != 0;
  float neg = 0.f;
  if (pos) {
    add_positive(P, n, [&](int lab) { return lg - (row[lab] - m); }, acc);
  } else {
    neg = lg - (row[C - 1] - m);
  }
  P.neg_ce[n] = neg;
  atomicAdd(&hist[key32(neg) >> 21], 1u);
}

__global__ void __launch_bounds__(kCeThreads, 1) ce_kernel(LossParams P, int warps_per_cta) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int C = P.C;
  const u32 tile_bytes = 32u * (u32)C * 4u;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float* bufs = reinterpret_cast<float*>(smem_raw);                                   // [warps][stages][32*C]
  u32* hist = reinterpret_cast<u32*>(smem_raw + (size_t)warps_per_cta * kStages * tile_bytes);
  u64* bars = reinterpret_cast<u64*>(hist + kBins);                                    // [warps][stages]
  double* red = reinterpret_cast<double*>(bars + kCeWarps * kStages);                  // [3][kCeWarps]

  for (int i = tid; i < kBins; i += kCeThreads) hist[i] = 0u;
  if (tid == 0) {
    for (int i = 0; i < warps_per_cta * kStages; ++i) mbar_init(&bars[i], 1);
    mbar_fence_init();
  }
  __syncthreads();

  CeAcc acc;
  acc.pos_ce = 0.f; acc.l1 = 0.f; acc.npos = 0;
  const long long full_tiles = P.N >> 5;
  if (warp < warps_per_cta) {
    const long long gw = (long long)blockIdx.x * warps_per_cta + warp;
    const long long stride = (long long)gridDim.x * warps_per_cta;
    float* mybuf = bufs + (size_t)warp * kStages * 32 * C;
    u64* mybar = bars + warp * kStages;
    const u64 pol = make_evict_first_policy();
    const char* src = reinterpret_cast<const char*>(P.pred_cls);
    // prologue
    if (lane == 0) {
      for (int s = 0; s < kStages; ++s) {
        long long t = gw + (long long)s * stride;
        if (t < full_tiles) {
          mbar_arrive_expect_tx(&mybar[s], tile_bytes);
          tma_load_1d_hint(mybuf + (size_t)s * 32 * C, src + (size_t)t * tile_bytes, tile_bytes, &mybar[s], pol);
        }
      }
    }
    int k = 0;
    for (long long t = gw; t < full_tiles; t += stride, ++k) {
      const int s = k % kStages;
      mbar_wait(&mybar[s], (u32)((k / kStages) & 1));
      const float* row = mybuf + (size_t)s * 32 * C + (size_t)lane * C;
      ce_one_prior(P, (t << 5) + lane, row, hist, acc);
      __syncwarp();
      const long long tn = t + (long long)kStages * stride;
      if (lane == 0 && tn < full_tiles) {
        mbar_arrive_expect_tx(&mybar[s], tile_bytes);
        tma_load_1d_hint(mybuf + (size_t)s * 32 * C, src + (size_t)tn * tile_bytes, tile_bytes, &mybar[s], pol);
      }
    }
    // tail rows (N % 32), plain loads, by the first warp of the grid
    const int tail = (int)(P.N & 31);
    if (gw == 0 && tail) {
      float* buf = mybuf;
      const float* g = P.pred_cls + (size_t)full_tiles * 32 * C;
      for (int i = lane; i < tail * C; i += 32) buf[i] = g[i];
      __syncwarp();
      if (lane < tail) ce_one_prior(P, (full_tiles << 5) + lane, buf + (size_t)lane * C, hist, acc);
    }
  }
  ce_pass_flush(P, acc, hist, red, tid);
}

// ---- the CE pass without the logits ----------------------------------------------------------------------
// When the softmax filter of the post-processing branch has already streamed the same logits (ssdg_detect_stage
// with row statistics), the loss needs no second pass over them: the background CE is there, and the positives
// (a few percent of the priors) gather their one ground-truth logit.  Same outputs as ce_kernel: the mining
// vector, its level-0 histogram, the per-CTA partial sums, the positives count.
__global__ void __launch_bounds__(kCeThreads) lossprep_kernel(LossParams P) {
  __shared__ u32 hist[kBins];
  __shared__ double red[3 * kCeWarps];
  const int tid = threadIdx.x;
  for (int i = tid; i < kBins; i += kCeThreads) hist[i] = 0u;
  __syncthreads();
  CeAcc acc;
  acc.pos_ce = 0.f; acc.l1 = 0.f; acc.npos = 0;
  const int C = P.C;
  auto one = [&](long long n, bool pos, float negbg) -> float {
    if (!pos) return negbg;
    add_positive(P, n, [&](int lab) {
      const float2 ml = P.row_ml[n];
      return ml.y - (__ldg(P.pred_cls + (size_t)n * C + lab) - ml.x);
    }, acc);
    return 0.f;
  };
  const long long gtid = (long long)blockIdx.x * kCeThreads + tid, gstride = (long long)gridDim.x * kCeThreads;
  const bool vec = (((uintptr_t)P.gt_mask) & 3) == 0 && (((uintptr_t)P.row_negbg | (uintptr_t)P.neg_ce) & 15) == 0;
  long long done = 0;
  if (vec) {
    const long long n4 = P.N >> 2;
    for (long long i = gtid; i < n4; i += gstride) {
      const uchar4 mk = reinterpret_cast<const uchar4*>(P.gt_mask)[i];
      const float4 nb = reinterpret_cast<const float4*>(P.row_negbg)[i];
      float4 o;
      o.x = one(4 * i, mk.x != 0, nb.x); o.y = one(4 * i + 1, mk.y != 0, nb.y);
      o.z = one(4 * i + 2, mk.z != 0, nb.z); o.w = one(4 * i + 3, mk.w != 0, nb.w);
      reinterpret_cast<float4*>(P.neg_ce)[i] = o;
      atomicAdd(&hist[key32(o.x) >> 21], 1u); atomicAdd(&hist[key32(o.y) >> 21], 1u);
      atomicAdd(&hist[key32(o.z) >> 21], 1u); atomicAdd(&hist[key32(o.w) >> 21], 1u);
    }
    done = n4 << 2;
  }
  for (long long n = done + gtid; n < P.N; n += gstride) {
    const float v = one(n, P.gt_mask[n] != 0, P.row_negbg[n]);
    P.neg_ce[n] = v;
    atomicAdd(&hist[key32(v) >> 21], 1u);
  }
  ce_pass_flush(P, acc, hist, red, tid);
}

// ---- radix select ------------------------------------------------------------------------------------
// Every CTA re-derives the state of the select from the (complete) histograms of the previous
// levels: prefix of the k-th key found so far and the rank still to resolve inside it.
struct SelectState {
  long long k;        // remaining rank inside the current prefix (1-based from the top)
  u32 prefix;         // key bits resolved so far (left-aligned per level)
  int status;
  double num_pos;
};

// Scan one histogram from the top: find bin with  count(bins above) < k <= count(bins >= bin).
// 256 threads, each owns nbins/256 consecutive bins (from the top) in registers: one round of global loads,
// a shuffle scan per warp and an 8-entry cross-warp prefix.
__device__ int scan_level(const u32* __restrict__ ghist, int nbins, long long& k, u32* sh /*[kBins]*/, int tid,
                          int* sh_bin, long long* sh_above) {
  const int per = nbins >> 8;   // 8 or 4
  const int hi = nbins - 1 - tid * per;
  u32 c[8];
  long long mine = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    c[j] = j < per ? ghist[hi - j] : 0u;
    mine += c[j];
  }
  long long incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long v = __shfl_up_sync(SSDG_FULL, incl, o);
    if ((tid & 31) >= o) incl += v;
  }
  long long* wtot = reinterpret_cast<long long*>(sh);   // [8] warp totals
  if ((tid & 31) == 31) wtot[tid >> 5] = incl;
  __syncthreads();
  long long above = incl - mine;
  for (int w = 0; w < (tid >> 5); ++w) above += wtot[w];
  if (above < k && k <= above + mine) {   // exactly one thread
    long long run = above;
    int bin = hi;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (j < per) {
        if (run + (long long)c[j] >= k) { bin = hi - j; break; }
        run += c[j];
      }
    }
    *sh_bin = bin;
    *sh_above = run;
  }
  __syncthreads();
  const int bin = *sh_bin;
  k -= *sh_above;
  __syncthreads();
  return bin;
}

__device__ void derive_state(const LossParams& P, int levels_done, SelectState& st, u32* sh, int tid, int* sh_bin,
                             long long* sh_above, double* sh_np) {
  if (tid < 32) {
    // counts are integers < 2^53: the sum is exact in any order
    double np = 0;
    const int n = (int)P.ws->nparts[0];
    for (int i = tid; i < n; i += 32) np += P.ws->part[i][2];
    np = warp_sum(np);
    if (tid == 0) { *sh_np = np; *sh_bin = 0; *sh_above = 0; }
  }
  __syncthreads();
  st.num_pos = P.global ? (double)P.ws->xnpos : *sh_np;
  st.k = (long long)P.ratio * (long long)st.num_pos;
  st.prefix = 0;
  st.status = 0;
  if (st.num_pos <= 0 || P.ratio <= 0) { st.status = SSDG_ERR_NO_POSITIVE; return; }
  if (st.k > P.N_all) { st.status = SSDG_ERR_TOPK_RANGE; return; }
  if (levels_done >= 1) st.prefix = (u32)scan_level(P.ws->hist[0], kBins, st.k, sh, tid, sh_bin, sh_above) << 21;
  if (levels_done >= 2) st.prefix |= (u32)scan_level(P.ws->hist[1], kBins, st.k, sh, tid, sh_bin, sh_above) << 10;
  if (levels_done >= 3) st.prefix |= (u32)scan_level(P.ws->hist[2], 1024, st.k, sh, tid, sh_bin, sh_above);
}

// level = 1: histogram bits 20..10 of keys whose bits 31..21 match; level = 2: bits 9..0.
__global__ void __launch_bounds__(256) select_kernel(LossParams P, int level) {
  __shared__ __align__(16) u32 sh[kBins];   // scan_level keeps 8-byte warp totals in its first words
  __shared__ int sh_bin;
  __shared__ long long sh_above;
  __shared__ double sh_np;
  pdl_wait();      // the previous level's histogram must be complete
  SelectState st;
  derive_state(P, level, st, sh, threadIdx.x, &sh_bin, &sh_above, &sh_np);
  if (st.status) return;
  for (int i = threadIdx.x; i < kBins; i += blockDim.x) sh[i] = 0u;
  __syncthreads();
  const u32 mask = level == 1 ? 0xffe00000u : 0xfffffc00u;
  const int shift = level == 1 ? 10 : 0;
  const u32 dmask = level == 1 ? 2047u : 1023u;
  const long long n4 = P.N >> 2;
  const float4* v4 = reinterpret_cast<const float4*>(P.neg_ce);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 v = v4[i];
    u32 k0 = key32(v.x), k1 = key32(v.y), k2 = key32(v.z), k3 = key32(v.w);
    if ((k0 & mask) == st.prefix) atomicAdd(&sh[(k0 >> shift) & dmask], 1u);
    if ((k1 & mask) == st.prefix) atomicAdd(&sh[(k1 >> shift) & dmask], 1u);
    if ((k2 & mask) == st.prefix) atomicAdd(&sh[(k2 >> shift) & dmask], 1u);
    if ((k3 & mask) == st.prefix) atomicAdd(&sh[(k3 >> shift) & dmask], 1u);
  }
  if (blockIdx.x == 0) {
    for (long long i = (n4 << 2) + threadIdx.x; i < P.N; i += blockDim.x) {
      u32 k0 = key32(P.neg_ce[i]);
      if ((k0 & mask) == st.prefix) atomicAdd(&sh[(k0 >> shift) & dmask], 1u);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kBins; i += blockDim.x) {
    u32 v = sh[i];
    if (v) atomicAdd(&P.ws->hist[level][i], v);
  }
}

__global__ void __launch_bounds__(256) final_kernel(LossParams P) {
  __shared__ __align__(16) u32 sh[kBins];
  __shared__ int sh_bin;
  __shared__ long long sh_above;
  __shared__ double sh_np;
  __shared__ double redd[8];
  __shared__ u32 redc[8], redo[8];
  __shared__ bool is_last;
  pdl_wait();      // the last level's histogram must be complete
  SelectState st;
  derive_state(P, 3, st, sh, threadIdx.x, &sh_bin, &sh_above, &sh_np);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const u32 kth = st.prefix;
  double sum = 0;
  u32 cnt = 0, ovl = 0;
  const long long gtid = (long long)blockIdx.x * blockDim.x + tid, gstride = (long long)gridDim.x * blockDim.x;
  const bool vec = (((uintptr_t)P.gt_mask | (uintptr_t)P.neg_mask) & 3) == 0;
  if (!st.status) {
    long long done = 0;
    if (vec) {   // four priors per thread per iteration: independent 16-byte / 4-byte loads in flight
      const long long n4 = P.N >> 2;
      const float4* v4 = reinterpret_cast<const float4*>(P.neg_ce);
      const uchar4* m4 = reinterpret_cast<const uchar4*>(P.gt_mask);
      for (long long i = gtid; i < n4; i += gstride) {
        const float4 v = v4[i];
        const uchar4 mk = m4[i];
        const bool n0 = key32(v.x) >= kth, n1 = key32(v.y) >= kth, n2 = key32(v.z) >= kth, n3 = key32(v.w) >= kth;
        sum += (double)((n0 ? v.x : 0.f) + (n1 ? v.y : 0.f)) + (double)((n2 ? v.z : 0.f) + (n3 ? v.w : 0.f));
        cnt += (u32)n0 + (u32)n1 + (u32)n2 + (u32)n3;
        ovl += (u32)(n0 && mk.x) + (u32)(n1 && mk.y) + (u32)(n2 && mk.z) + (u32)(n3 && mk.w);
        if (P.neg_mask) reinterpret_cast<uchar4*>(P.neg_mask)[i] = make_uchar4(n0, n1, n2, n3);
      }
      done = n4 << 2;
    }
    for (long long i = done + gtid; i < P.N; i += gstride) {
      const float v = P.neg_ce[i];
      const bool neg = key32(v) >= kth;
      if (neg) {
        sum += (double)v;
        cnt += 1;
        if (P.gt_mask[i]) ovl += 1;
      }
      if (P.neg_mask) P.neg_mask[i] = neg ? 1 : 0;
    }
  } else if (P.neg_mask) {
    for (long long i = gtid; i < P.N; i += gstride) P.neg_mask[i] = 0;
  }
  sum = warp_sum(sum);
  cnt = __reduce_add_sync(SSDG_FULL, cnt);
  ovl = __reduce_add_sync(SSDG_FULL, ovl);
  if (lane == 0) { redd[warp] = sum; redc[warp] = cnt; redo[warp] = ovl; }
  __syncthreads();
  if (tid == 0) {
    double s = 0; u32 c = 0, o = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { s += redd[w]; c += redc[w]; o += redo[w]; }
    P.ws->fpart[blockIdx.x][0] = s;
    P.ws->fcount[blockIdx.x][0] = c;
    P.ws->fcount[blockIdx.x][1] = o;
    __threadfence();
    is_last = atomicAdd(&P.ws->ticket[0], 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  // deterministic final reduction: fixed assignment of partials to threads, fixed tree
  double s_pos = 0, s_l1 = 0, s_neg = 0;
  unsigned long long n_neg = 0, n_ovl = 0;
  const int np = (int)P.ws->nparts[0];
  for (int i = tid; i < np; i += blockDim.x) { s_pos += P.ws->part[i][0]; s_l1 += P.ws->part[i][1]; }
  for (int i = tid; i < (int)gridDim.x; i += blockDim.x) {
    s_neg += ((volatile double*)P.ws->fpart[i])[0];
    n_neg += ((volatile u32*)P.ws->fcount[i])[0];
    n_ovl += ((volatile u32*)P.ws->fcount[i])[1];
  }
  __shared__ double fin[5][8];
  s_pos = warp_sum(s_pos); s_l1 = warp_sum(s_l1); s_neg = warp_sum(s_neg);
  double d_neg = warp_sum((double)n_neg), d_ovl = warp_sum((double)n_ovl);
  if (lane == 0) { fin[0][warp] = s_pos; fin[1][warp] = s_l1; fin[2][warp] = s_neg; fin[3][warp] = d_neg; fin[4][warp] = d_ovl; }
  __syncthreads();
  if (tid != 0) return;
  s_pos = s_l1 = s_neg = d_neg = d_ovl = 0;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
    s_pos += fin[0][w]; s_l1 += fin[1][w]; s_neg += fin[2][w]; d_neg += fin[3][w]; d_ovl += fin[4][w];
  }
  n_neg = (unsigned long long)d_neg; n_ovl = (unsigned long long)d_ovl;
  double* r = P.result;
  int status = st.status;
  const u32 n_badlab = ((volatile u32*)P.ws->nparts)[1];
  if (!status && n_ovl) status = SSDG_ERR_POS_NEG_OVERLAP;  // models/ssd_model.py:375 (positives mined as negatives)
  if (!status && n_badlab) status = SSDG_ERR_LABEL_RANGE;
  const double nan = CUDART_NAN;
  const double l_pos = status ? nan : s_pos / st.num_pos;
  const double l_neg = status ? nan : s_neg / (double)n_neg;
  const double l_loc = status ? nan : s_l1 / st.num_pos;
  r[0] = (l_loc + l_pos) + l_neg;  // models/ssd_model.py:396
  r[1] = l_pos; r[2] = l_neg; r[3] = l_loc;
  r[4] = st.num_pos; r[5] = (double)n_neg;
  r[6] = status ? nan : (double)unkey32(kth);
  r[7] = (double)status;
  r[8] = s_pos; r[9] = s_neg; r[10] = s_l1;
  r[11] = sh_np;   // this shard's own positives (== r[4] unless the mining is cross-shard)
  // data-dependent errors seen by THIS shard (overlap :375, label range): additive, so a cross-shard caller sums it
  // with [8..11] and every shard agrees on success
  r[12] = (double)n_ovl + (double)n_badlab;
  for (int i = 13; i < SSDG_LOSS_RESULT_LEN; ++i) r[i] = 0;
}

// ---- gradient (models/ssd_model.py:248 through :355-386) ---------------------------------------------
//   d/d logits = softmax * (pos/Npos + neg/Nneg) - onehot(gt)*pos/Npos - onehot(bg)*neg/Nneg
//   d/d pred_box = sign(pred - gt) * pos/Npos
// The output is as large as the logits but only the positives and the mined negatives (a few percent of the rows each)
// are non-zero: the array is zero-filled by a stream-ordered memset (write bandwidth, no read of the logits), and this
// kernel then visits the non-zero rows only -- one warp per group of 32 priors finds them by ballot and computes them
// row by row, the loads of up to four rows in flight at once.
constexpr int kGradThreads = 256;

__global__ void __launch_bounds__(kGradThreads) grad_kernel(LossParams P) {
  const double* r = P.result;
  const bool bad = r[7] != 0.0 || r[12] != 0.0;
  const float wpos = bad ? CUDART_NAN_F : (float)(1.0 / r[4]);
  const float wneg = bad ? CUDART_NAN_F : (float)(1.0 / r[5]);
  const u32 kth = key32((float)r[6]);
  const int C = P.C;
  const int lane = threadIdx.x & 31;
  const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
  const long long groups = (P.N + 31) >> 5;
  constexpr int kRows = 4;     // rows whose logits are loaded together
  constexpr int kPer = 4;      // classes per lane held in registers (C <= 128; more classes take the plain loop)
  for (long long g = gw; g < groups; g += nw) {
    const long long n = (g << 5) + lane;
    const bool in = n < P.N;
    const bool pos = in && P.gt_mask[n] != 0;
    const bool neg = in && !bad && key32(P.neg_ce[n]) >= kth;
    if (in) {   // lane = row: d / d pred_box
      float4 gb4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (pos) {
        const float4 pb = __ldg(reinterpret_cast<const float4*>(P.pred_box) + n);
        const float4 gb = __ldg(reinterpret_cast<const float4*>(P.gt_box) + n);
        auto sg = [&](float d) { return d > 0.f ? wpos : (d < 0.f ? -wpos : 0.f); };
        gb4 = make_float4(sg(pb.x - gb.x), sg(pb.y - gb.y), sg(pb.z - gb.z), sg(pb.w - gb.w));
      }
      reinterpret_cast<float4*>(P.grad_box)[n] = gb4;
    }
    int lab = pos ? P.gt_cls[n] : 0;
    lab = lab < 0 ? 0 : (lab >= C ? C - 1 : lab);   // (out-of-range labels make the whole result `bad`)
    u32 act = __ballot_sync(SSDG_FULL, in && (pos || neg || bad));
    while (act) {
      int rows[kRows];
      int nr = 0;
#pragma unroll
      for (int k = 0; k < kRows; ++k) {
        rows[k] = -1;
        if (act) { rows[k] = __ffs(act) - 1; act &= act - 1; ++nr; }
      }
      if (C <= 32 * kPer) {
        float x[kRows][kPer];
#pragma unroll
        for (int k = 0; k < kRows; ++k) {
          const float* src = P.pred_cls + (size_t)((g << 5) + (rows[k] < 0 ? 0 : rows[k])) * C;
#pragma unroll
          for (int q = 0; q < kPer; ++q) {
            const int c = lane + 32 * q;
            x[k][q] = (rows[k] >= 0 && c < C) ? __ldg(src + c) : -CUDART_INF_F;
          }
        }
#pragma unroll
        for (int k = 0; k < kRows; ++k) {
          if (rows[k] < 0) break;      // warp-uniform
          const int rr = rows[k];
          const bool rp = __shfl_sync(SSDG_FULL, (int)pos, rr) != 0, rn = __shfl_sync(SSDG_FULL, (int)neg, rr) != 0;
          const int rl = __shfl_sync(SSDG_FULL, lab, rr);
          float m = fmaxf(fmaxf(x[k][0], x[k][1]), fmaxf(x[k][2], x[k][3]));
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(SSDG_FULL, m, o));
          float e[kPer], sum = 0.f;
#pragma unroll
          for (int q = 0; q < kPer; ++q) { e[q] = __expf(x[k][q] - m); sum += e[q]; }   // exp(-inf) = 0 beyond C
          sum = warp_sum(sum);
          const float w = (rp ? wpos : 0.f) + (rn ? wneg : 0.f);
          const float inv = w / sum;
          float* dst = P.grad_cls + (size_t)((g << 5) + rr) * C;
#pragma unroll
          for (int q = 0; q < kPer; ++q) {
            const int c = lane + 32 * q;
            if (c < C) {
              float v = e[q] * inv;
              if (rp && c == rl) v -= wpos;
              if (rn && c == C - 1) v -= wneg;
              __stcs(&dst[c], v);
            }
          }
        }
      } else {
        for (int k = 0; k < nr; ++k) {
          const int rr = rows[k];
          const bool rp = __shfl_sync(SSDG_FULL, (int)pos, rr) != 0, rn = __shfl_sync(SSDG_FULL, (int)neg, rr) != 0;
          const int rl = __shfl_sync(SSDG_FULL, lab, rr);
          const float* x = P.pred_cls + (size_t)((g << 5) + rr) * C;
          float m = -CUDART_INF_F;
          for (int c = lane; c < C; c += 32) m = fmaxf(m, x[c]);
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(SSDG_FULL, m, o));
          float sum = 0.f;
          for (int c = lane; c < C; c += 32) sum += __expf(x[c] - m);
          sum = warp_sum(sum);
          const float inv = ((rp ? wpos : 0.f) + (rn ? wneg : 0.f)) / sum;
          float* dst = P.grad_cls + (size_t)((g << 5) + rr) * C;
          for (int c = lane; c < C; c += 32) {
            float v = __expf(x[c] - m) * inv;
            if (rp && c == rl) v -= wpos;
            if (rn && c == C - 1) v -= wneg;
            __stcs(&dst[c], v);
          }
        }
      }
    }
  }
}

// Shared memory for the tile rings of a ce_kernel CTA: all kCeWarps warps up to C = 100, fewer beyond.  The warp count
// decides how tiles map to CTAs, and so how the per-CTA partial sums are grouped: changing it changes the loss bits.
constexpr size_t kCeSmemBudget = 200 * 1024;

static int ce_warps_for(int C) {
  size_t per_warp = (size_t)kStages * 32 * C * 4;
  int w = (int)(kCeSmemBudget / per_warp);
  if (w > kCeWarps) w = kCeWarps;
  return w;
}
static size_t ce_smem_bytes(int C, int warps) {
  return (size_t)warps * kStages * 32 * C * 4 + kBins * 4 + kCeWarps * kStages * 8 + 3 * kCeWarps * 8 + 128;
}

}  // namespace ssdg

using namespace ssdg;

extern "C" size_t ssdg_loss_workspace_bytes(int64_t batch, int32_t n_priors, int32_t n_classes) {
  (void)n_classes;
  if (batch <= 0 || n_priors <= 0) return 0;
  return align_up(sizeof(LossWs), 256) + align_up((size_t)batch * n_priors * 4, 256);
}

// The stages one loss_run call enqueues, a bit set; stage k of ssdg_multibox_loss_stage is bit k.  Between the stages
// of a cross-shard run the caller sums the exchange words over the shards.
constexpr int kStageCe = 1;                         // CE pass (+ level-0 histogram, positives count)
constexpr int kStageLevel1 = 2, kStageLevel2 = 4;   // radix levels 1 and 2
constexpr int kStageFinal = 8;                      // mask, sums, result
constexpr int kStageGrad = 16;                      // gradient: in a cross-shard run AFTER the last exchange
                                                    // (it reads the global num_neg from the result block)
constexpr int kStageAll = kStageCe | kStageLevel1 | kStageLevel2 | kStageFinal | kStageGrad;

static int loss_run(int stages, int global, long long n_all, const float* row_ml, const float* row_negbg,
                    const int32_t* gt_cls, const float* gt_box,
                    const uint8_t* gt_mask, const float* pred_box, const float* pred_cls, int64_t batch,
                    int32_t n_priors, int32_t n_classes, int32_t neg_ratio, double* out_result, uint8_t* out_neg_mask,
                    float* out_neg_ce, float* grad_box, float* grad_cls, void* workspace, size_t workspace_bytes,
                    void* stream) {
  if (!gt_cls || !gt_box || !gt_mask || !pred_box || !pred_cls || !out_result) return SSDG_ERR_ARG;
  if (batch <= 0 || n_priors <= 0 || n_classes < 2 || neg_ratio <= 0) return SSDG_ERR_ARG;
  if ((grad_box == nullptr) != (grad_cls == nullptr)) return SSDG_ERR_ARG;
  if (((uintptr_t)pred_cls | (uintptr_t)pred_box | (uintptr_t)gt_box | (uintptr_t)out_neg_ce) & 15) return SSDG_ERR_ALIGN;
  if (!workspace || ((uintptr_t)workspace & 255) || workspace_bytes < ssdg_loss_workspace_bytes(batch, n_priors, n_classes))
    return SSDG_ERR_WORKSPACE;
  const int warps = ce_warps_for(n_classes);
  if (warps < 1) return SSDG_ERR_LIMIT;
  cudaStream_t st = (cudaStream_t)stream;
  LossParams P;
  P.gt_cls = gt_cls; P.gt_box = gt_box; P.gt_mask = gt_mask; P.pred_box = pred_box; P.pred_cls = pred_cls;
  P.N = (long long)batch * n_priors; P.C = n_classes; P.ratio = neg_ratio;
  P.N_all = global ? n_all : P.N; P.global = global;
  if ((row_ml == nullptr) != (row_negbg == nullptr)) return SSDG_ERR_ARG;
  if (((uintptr_t)row_ml & 7) || ((uintptr_t)row_negbg & 3)) return SSDG_ERR_ALIGN;
  P.row_ml = reinterpret_cast<const float2*>(row_ml); P.row_negbg = row_negbg;
  if (P.N_all < P.N) return SSDG_ERR_ARG;
  P.ws = (LossWs*)workspace;
  P.neg_ce = out_neg_ce ? out_neg_ce : (float*)((unsigned char*)workspace + align_up(sizeof(LossWs), 256));
  P.neg_mask = out_neg_mask; P.result = out_result; P.grad_box = grad_box; P.grad_cls = grad_cls;
  if (stages & kStageCe) {
    SSDG_CUDA_TRY(cudaMemsetAsync(&P.ws->hist[0][0], 0, sizeof(LossWs) - offsetof(LossWs, hist), st));
    prof_begin(SSDG_PROF_CE, st);
    if (row_ml) {
      int grid = (int)((P.N / 4 + 255) / 256);
      if (grid > 256) grid = 256;   // LossWs::part
      if (grid < 1) grid = 1;
      SSDG_CUDA_TRY(cudaFuncSetAttribute(lossprep_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
      lossprep_kernel<<<grid, kCeThreads, 0, st>>>(P);
    } else {
      const size_t smem = ce_smem_bytes(n_classes, warps);
      SSDG_CUDA_TRY(cudaFuncSetAttribute(ce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      int grid = sm_count();
      if (grid > 256) grid = 256;
      const long long tiles = (P.N + 31) / 32;
      const long long need = (tiles + warps - 1) / warps;
      if (need < grid) grid = (int)need;
      ce_kernel<<<grid, kCeThreads, smem, st>>>(P, warps);
    }
    prof_end(SSDG_PROF_CE, st);
    SSDG_LAUNCH_CHECK();
  }
  int sgrid = sm_count() * 4;
  const long long sneed = (P.N / 4 + 255) / 256;
  if (sneed < sgrid) sgrid = (int)(sneed > 0 ? sneed : 1);
  if (sgrid > 1024) sgrid = 1024;
  if (stages & (kStageLevel1 | kStageLevel2)) {
    prof_begin(SSDG_PROF_LOSS_TAIL, st);
    SSDG_CUDA_TRY(cudaFuncSetAttribute(select_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    if (stages & kStageLevel1) SSDG_CUDA_TRY(launch_pdl(select_kernel, dim3(sgrid), dim3(256), 0, st, P, 1));
    if (stages & kStageLevel2) SSDG_CUDA_TRY(launch_pdl(select_kernel, dim3(sgrid), dim3(256), 0, st, P, 2));
    SSDG_LAUNCH_CHECK();
  }
  if (stages & kStageFinal) {
    SSDG_CUDA_TRY(cudaFuncSetAttribute(final_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    SSDG_CUDA_TRY(launch_pdl(final_kernel, dim3(sgrid), dim3(256), 0, st, P));
    prof_end(SSDG_PROF_LOSS_TAIL, st);
    SSDG_LAUNCH_CHECK();
  }
  if ((stages & kStageGrad) && grad_cls) {
    prof_begin(SSDG_PROF_GRAD, st);
    SSDG_CUDA_TRY(cudaMemsetAsync(grad_cls, 0, (size_t)P.N * n_classes * sizeof(float), st));
    {
      int ggrid = sm_count() * 8;
      const long long gneed = (((P.N + 31) >> 5) * 32 + kGradThreads - 1) / kGradThreads;
      if (gneed < ggrid) ggrid = (int)(gneed > 0 ? gneed : 1);
      grad_kernel<<<ggrid, kGradThreads, 0, st>>>(P);
    }
    prof_end(SSDG_PROF_GRAD, st);
    SSDG_LAUNCH_CHECK();
  }
  return SSDG_OK;
}

extern "C" int ssdg_multibox_loss(const int32_t* gt_cls, const float* gt_box, const uint8_t* gt_mask,
                                  const float* pred_box, const float* pred_cls, int64_t batch, int32_t n_priors,
                                  int32_t n_classes, int32_t neg_ratio, double* out_result, uint8_t* out_neg_mask,
                                  float* out_neg_ce, float* grad_box, float* grad_cls, void* workspace,
                                  size_t workspace_bytes, void* stream) {
  return loss_run(kStageAll, 0, 0, nullptr, nullptr, gt_cls, gt_box, gt_mask, pred_box, pred_cls, batch, n_priors,
                  n_classes, neg_ratio, out_result, out_neg_mask, out_neg_ce, grad_box, grad_cls, workspace,
                  workspace_bytes, stream);
}

extern "C" int ssdg_multibox_loss_stage(int32_t stage, int64_t global_priors, const float* row_ml,
                                        const float* row_negbg, const int32_t* gt_cls,
                                        const float* gt_box, const uint8_t* gt_mask, const float* pred_box,
                                        const float* pred_cls, int64_t batch, int32_t n_priors, int32_t n_classes,
                                        int32_t neg_ratio, double* out_result, uint8_t* out_neg_mask,
                                        float* out_neg_ce, float* grad_box, float* grad_cls, void* workspace,
                                        size_t workspace_bytes, void* stream) {
  if (stage < 0 || stage > 4 || global_priors <= 0) return SSDG_ERR_ARG;
  if (stage == 4 && !grad_cls) return SSDG_ERR_ARG;
  return loss_run(1 << stage, 1, global_priors, row_ml, row_negbg, gt_cls, gt_box, gt_mask, pred_box, pred_cls, batch, n_priors,
                  n_classes, neg_ratio, out_result, out_neg_mask, out_neg_ce, grad_box, grad_cls, workspace,
                  workspace_bytes, stream);
}

extern "C" int ssdg_multibox_loss_fused(const float* row_ml, const float* row_negbg, const int32_t* gt_cls,
                                        const float* gt_box, const uint8_t* gt_mask, const float* pred_box,
                                        const float* pred_cls, int64_t batch, int32_t n_priors, int32_t n_classes,
                                        int32_t neg_ratio, double* out_result, uint8_t* out_neg_mask,
                                        float* out_neg_ce, float* grad_box, float* grad_cls, void* workspace,
                                        size_t workspace_bytes, void* stream) {
  if (!row_ml || !row_negbg) return SSDG_ERR_ARG;
  return loss_run(kStageAll, 0, 0, row_ml, row_negbg, gt_cls, gt_box, gt_mask, pred_box, pred_cls, batch, n_priors,
                  n_classes, neg_ratio, out_result, out_neg_mask, out_neg_ce, grad_box, grad_cls, workspace,
                  workspace_bytes, stream);
}

extern "C" int ssdg_loss_exchange(void* workspace, int32_t which, void** out_ptr, int64_t* out_count) {
  if (!workspace || !out_ptr || !out_count || which < 0 || which > 3) return SSDG_ERR_ARG;
  LossWs* ws = (LossWs*)workspace;
  if (which < 3) { *out_ptr = &ws->hist[which][0]; *out_count = kBins; }     // int32 counts
  else { *out_ptr = &ws->xnpos; *out_count = 1; }                           // int64 count
  return SSDG_OK;
}
