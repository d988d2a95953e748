// nms.cuh — exact greedy NMS for one segment (image) per CTA.  Included by nms.cu (generic C-ABI entry),
// yolo_decode.cu and effdet.cu (fused post-processing).  The candidate store those two share — its workspace layout, the
// append of the filter kernels and the output tail of the finalize kernels — is at the end of this file (CandStore).
//
// Replaces the tf.while_loop NMS drivers of the reference:
//   utils/tf_iou_utils.py:67-108   GetIOUNMS            (class-agnostic, survivor iff metric <  thr; NaN drops)
//   utils/tf_iou_utils.py:110-157  GetIOUNMSByClasses   (suppressed iff metric >= thr and same class; NaN stays)
//   efficientnet/utils/nms.py:5-61 get_nms              (GetIOUNMS + stop at first top score < score_threshold)
// Semantics reproduced exactly: candidates ordered by (score descending, index ascending) as tf.argsort
// (DESCENDING) does; candidate j is emitted iff no earlier *emitted* i suppresses it; at most max_out emitted.
//
// Algorithm (B200: one 1024-thread CTA per image, everything after the score read lives in shared memory):
//   1. top-window selection by radix buckets of the 64-bit key (~ordered(score) << 32 | order_id): one pass finds
//      the range of the eligible keys, a second one histograms them into 2048 buckets of that range (monotone in the
//      key), a prefix scan picks the bucket where the cumulative count reaches the window target, a third pass
//      gathers every key up to that bucket into shared memory — an exact top-k cut with no sorting at all.  The
//      gathered window (<= 4096 keys) is then ordered in place by the same trick applied to its own range: 2048
//      buckets, a per-bucket chain, rank inside the chain (chains hold ~1-2 keys), exclusive scan -> the exact global
//      order of its members as an index array.  (The sampled-pivot + bitonic path of round 1 — 66 + 78 barrier stages
//      — is kept only as the fallback for a bucket that alone overflows the window, e.g. thousands of equal scores.)
//      Segments with <= 4096 candidates are gathered whole;
//      Segments of at most 8 keys per thread whose caller opts in (YOLO) read their scores once and run the passes
//      from registers; segments above 8192 keys take the bucket range from one sample per thread (the buckets are
//      monotone whatever the bounds, so the cut stays exact) and the count from the histogram pass;
//   2. class-agnostic mode: the sorted window is consumed lazily in tiles of 64 candidates: a tile is first tested
//      against every box emitted so far (kept list in shared memory; 64 x n_kept pairs spread over the 1024 threads),
//      then resolved internally with a 64x64 ballot bitmask and a one-warp fixed-point sweep (skipped when the tile has
//      no internal conflict).  Only as many tiles as are needed to emit max_out boxes are touched, so the work is
//      O(emitted^2) and independent of the window size;
//   3. per-class mode: a chunk of 1024 ranked candidates is split stably by class bucket; all pairs (i < j) of all
//      buckets form one flat index space that the threads share equally (bit i of member j's word = "i suppresses
//      j"), one thread per bucket then walks its members in rank order with the alive set in a register, and the
//      survivors are emitted in rank order.
// Every pair test starts with bm_surely_below (boxmath.cuh): no overlap, or IoU clearly below the threshold by a
// division-free comparison — the full metric (2-4 IEEE divisions) runs for ~1 pair in 3000 on dense heads.
// The metric is a template parameter so each instantiation carries one metric's code (the 7-way runtime switch
// inlined at three call sites was 150 KB of SASS and did not fit the instruction cache).
#pragma once
#include "boxmath.cuh"
#include "common.cuh"

#define NMS_THREADS 1024
#define NMS_CHUNK 1024
#define NMS_WINDOW 4096
#define NMS_SAMPLES 2048
#define NMS_TARGET 1536
#define NMS_MAX_OUT_LIMIT 4096

struct NmsSegment {
  const float* boxes;        // [n,4] in the metric family's corner order
  const float* scores;       // [n]
  const int32_t* classes;    // [n] or nullptr (required for BY_CLASS)
  const uint32_t* order_id;  // [n] unique tie-break ids (ascending = earlier) or nullptr -> position
  int n;
};

// Optional pre-gathered first window of a segment (produced by nms_preselect_kernel with several CTAs per
// segment, for segments too large for one CTA to scan quickly).  Ignored unless its counters show a valid window.
struct NmsPre {
  const unsigned long long* keys;  // [NMS_PRE_CAP]
  const uint32_t* pos;             // [NMS_PRE_CAP]
  const int* count;                // gathered (may exceed NMS_PRE_CAP: then invalid)
  const int* eligible;             // eligible candidates in the whole segment
  const unsigned long long* khi;   // pivot used
};

struct NmsConfig {
  int metric;
  int mode;
  float iou_thr;
  float score_thr;
  int use_score_thr;
  int max_out;
};

__host__ __device__ inline size_t nms_smem_bytes(int max_out) {
  // window keys 32K + window pos 16K + samples 16K + cand 28K + class-bucket heads 1K + kept 32B*max_out + small
  return (size_t)NMS_WINDOW * 12 + (size_t)NMS_SAMPLES * 8 + NMS_CHUNK * 28 + 256 * 4 + (size_t)max_out * 32 + 1024;
}

// Large segments pay full passes over their scores per extra window, so they take big windows (ordering a window by
// buckets is cheap, and only the part that is needed is ever consumed).
#define NMS_PRE_MIN_N 65536      // segments above this get their first window from the multi-CTA pre-selection
#define NMS_TARGET_LARGE 3072
#define NMS_PRE_CAP 8192          // capacity of a pre-gathered list (keys below a sampled pivot aiming at NMS_TARGET_LARGE)
__host__ __device__ inline int nms_window_target(int max_out, int n) {
  if (n > NMS_PRE_MIN_N) return NMS_TARGET_LARGE;
  if (n > 16384) return NMS_TARGET;
  int t = max_out + (max_out >> 1);
  if (t < 512) t = 512;
  if (t > NMS_TARGET) t = NMS_TARGET;
  return t;
}

__device__ __forceinline__ uint32_t nms_dkey(float s) {
  uint32_t u = __float_as_uint(s);
  if ((u << 1) == 0u) u = 0u;  // -0 == +0 for tf.argsort
  uint32_t k = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ~k;  // ascending dkey == descending score
}

template <int METRIC>
__device__ __forceinline__ bool nms_suppresses(const BoxT& kept, int kept_cls, const BoxT& cand, int cand_cls, int mode,
                                                float thr) {
  if (mode == B200_NMS_BY_CLASS) {
    if (kept_cls != cand_cls) return false;
    if (bm_surely_below(kept, cand, METRIC, thr)) return false;
    return bm_metric(kept, cand, METRIC) >= thr;
  }
  if (bm_surely_below(kept, cand, METRIC, thr)) return false;
  return !(bm_metric(kept, cand, METRIC) < thr);
}

// ascending bitonic sort of sK[0..npad) (npad a power of two) with optional payload sP, whole CTA.
// (A register/shuffle variant with ~3x fewer block barriers was measured slower: every element then does its own
// compare, twice the ALU work of the pairwise exchange below, and the barriers were not the bottleneck.)
template <int THREADS = NMS_THREADS>
__device__ __forceinline__ void nms_bitonic(unsigned long long* sK, uint32_t* sP, int npad) {
  for (int k = 2; k <= npad; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < npad; t += THREADS) {
        const int ixj = t ^ j;
        if (ixj > t) {
          const unsigned long long a = sK[t], b = sK[ixj];
          const bool asc = ((t & k) == 0);
          if ((a > b) == asc) {
            sK[t] = b; sK[ixj] = a;
            if (sP) { const uint32_t pa = sP[t]; sP[t] = sP[ixj]; sP[ixj] = pa; }
          }
        }
      }
      __syncthreads();
    }
  }
}

#define NMS_BINS 2048
#define NMS_KC 8   // keys a thread keeps in registers for the selection passes of a small segment
#define NMS_LOADS 4   // independent loads a thread keeps in flight in a selection pass over a large segment (8: no faster, spills)

// bucket of a descending-score key inside [dmin, dmax]: monotone non-decreasing in d (int->float rounding, the
// multiplication by a positive constant and the truncation all are), so bucket(a) < bucket(b) implies a < b
// (keys below dmin fall into bucket 0, keys above dmax into the last one: dmin / dmax may be estimates from a sample)
__device__ __forceinline__ int nms_bin(uint32_t d, uint32_t dmin, float scale) {
  const int b = (int)((float)(d - dmin) * scale);   // the conversion saturates
  return d <= dmin ? 0 : (b < NMS_BINS - 1 ? b : NMS_BINS - 1);
}
__device__ __forceinline__ float nms_bin_scale(uint32_t dmin, uint32_t dmax) {
  return (float)NMS_BINS / ((float)(dmax - dmin) + 1.0f);
}

// CTA-wide (min, max, sum) of three per-thread values; red = 3 * 32 uint32 of scratch.  All threads get the result.
template <int THREADS>
__device__ __forceinline__ void nms_block_minmaxsum(uint32_t& mn, uint32_t& mx, int& sum, uint32_t* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    sum += __shfl_xor_sync(0xffffffffu, sum, o);
  }
  if (lane == 0) { red[warp] = mn; red[32 + warp] = mx; red[64 + warp] = (uint32_t)sum; }
  __syncthreads();
  mn = 0xffffffffu; mx = 0u; sum = 0;
#pragma unroll
  for (int w = 0; w < THREADS / 32; ++w) { mn = min(mn, red[w]); mx = max(mx, red[32 + w]); sum += (int)red[64 + w]; }
  __syncthreads();
}

// In-place exclusive prefix sum of hist[NMS_BINS] by the whole CTA.  Returns the total; when `target` > 0 also reports
// through *cut_out (shared) the first bucket whose inclusive count reaches target (NMS_BINS - 1 when none does).
template <int THREADS>
__device__ __forceinline__ int nms_block_scan_bins(int* hist, uint32_t* red, int target, int* cut_out) {
  constexpr int PER = NMS_BINS / THREADS;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int v[PER], local = 0;
#pragma unroll
  for (int k = 0; k < PER; ++k) { v[k] = hist[threadIdx.x * PER + k]; local += v[k]; }
  int incl = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
  if (lane == 31) red[warp] = (uint32_t)incl;
  if (threadIdx.x == 0 && cut_out) *cut_out = NMS_BINS - 1;
  __syncthreads();
  int base = 0, total = 0;
#pragma unroll
  for (int w = 0; w < THREADS / 32; ++w) { const int t = (int)red[w]; if (w < warp) base += t; total += t; }
  int run = base + incl - local;
#pragma unroll
  for (int k = 0; k < PER; ++k) {
    hist[threadIdx.x * PER + k] = run;
    if (cut_out && target > 0 && run < target && run + v[k] >= target) *cut_out = threadIdx.x * PER + k;
    run += v[k];
  }
  __syncthreads();
  return total;
}

// Exact ascending order of keys[0..n) (n <= NMS_WINDOW, 64-bit keys in shared memory; ties by position) as an index array:
// ord[r] = position of the r-th smallest key.  bins: 2 * NMS_BINS ints of scratch (ord may alias its first half),
// nxt: n ints of scratch, red: 96 uint32.  Cost: a handful of barriers and O(chain length) per key.
// With have_range the caller supplies mn <= every key's high word and an estimate mx of the largest one (keys above mx all
// fall into the last bucket — still monotone, so the order stays exact) and the range pass with its two barriers is skipped.
template <int THREADS>
__device__ __forceinline__ void nms_bucket_order(const unsigned long long* keys, int n, int* bins, int* nxt, uint32_t* red,
                                                 unsigned short* ord, bool have_range = false, uint32_t mn_in = 0u,
                                                 uint32_t mx_in = 0u) {
  constexpr int PER = NMS_WINDOW / THREADS;
  int* hist = bins;
  int* head = bins + NMS_BINS;
  uint32_t mn = 0xffffffffu, mx = 0u;
  int dummy = 0;
  if (!have_range) {
    for (int t = threadIdx.x; t < n; t += THREADS) {
      const uint32_t d = (uint32_t)(keys[t] >> 32);
      mn = min(mn, d); mx = max(mx, d);
    }
  }
  for (int b = threadIdx.x; b < NMS_BINS; b += THREADS) { hist[b] = 0; head[b] = -1; }
  if (have_range) { mn = mn_in; mx = mx_in < mn_in ? mn_in : mx_in; __syncthreads(); }
  else nms_block_minmaxsum<THREADS>(mn, mx, dummy, red);   // its barriers also publish the cleared bins
  const float scale = nms_bin_scale(mn, mx);
  for (int t = threadIdx.x; t < n; t += THREADS) {
    const int b = nms_bin((uint32_t)(keys[t] >> 32), mn, scale);
    atomicAdd(&hist[b], 1);
    nxt[t] = atomicExch(&head[b], t);
  }
  __syncthreads();
  nms_block_scan_bins<THREADS>(hist, red, 0, nullptr);
  int dst[PER];
#pragma unroll
  for (int u = 0; u < PER; ++u) {
    const int t = (int)threadIdx.x + u * THREADS;
    dst[u] = 0;
    if (t < n) {
      const unsigned long long K = keys[t];
      const int b = nms_bin((uint32_t)(K >> 32), mn, scale);
      int r = 0;
      for (int j = head[b]; j >= 0; j = nxt[j]) {  // equal keys (only the ineligible-sample sentinel repeats) order by position
        const unsigned long long Kj = keys[j];
        r += (Kj < K || (Kj == K && j < t)) ? 1 : 0;
      }
      dst[u] = hist[b] + r;
    }
  }
  __syncthreads();   // every chain walk is finished: the bins may be overwritten by ord
#pragma unroll
  for (int u = 0; u < PER; ++u) {
    const int t = (int)threadIdx.x + u * THREADS;
    if (t < n) ord[dst[u]] = (unsigned short)t;
  }
  __syncthreads();
}

// Runs NMS for one segment with the whole CTA (blockDim.x == THREADS).  out_pos receives the local
// positions (0..n-1) of emitted candidates in emit order; returns the number emitted (uniform across threads).
// How a candidate's box is obtained when it enters the window: by default a read of seg.boxes; a caller may decode
// it on demand instead (YOLO: only the few hundred candidates NMS actually looks at are ever decoded).
struct NmsLoadDirect {
  static constexpr bool kKeyCache = false;   // register cache of a small segment's keys (16 registers): opt-in per caller
  static constexpr int kMode = -1;           // -1: NmsConfig::mode decides at run time; else the caller's only mode (the other
                                             // mode's code — and its registers — are not compiled into that kernel)
  static constexpr bool kSampleRange = true; // large segments: bucket range from a sample instead of a full pass (compiled out for
                                             // the YOLO kernels: their segments are small, and the mere presence of the path cost
                                             // the single-image kernel 2.6 us, measured)
  __device__ __forceinline__ float4 operator()(const NmsSegment& seg, uint32_t pos) const {
    return __ldg(reinterpret_cast<const float4*>(seg.boxes) + pos);
  }
};

struct NmsLoadDirectAgnostic : NmsLoadDirect {   // callers that only ever run class-agnostic NMS (EfficientDet)
  static constexpr int kMode = B200_NMS_AGNOSTIC;
};

// THREADS = CTA size (a multiple of 64, <= NMS_THREADS): 1024 for the lowest per-image latency; 512 lets two CTAs
// share an SM (64 registers/thread), which is faster for batches that do not fit one CTA per SM.
template <int METRIC, class BoxLoad = NmsLoadDirect, int THREADS = NMS_THREADS>
static __device__ int nms_run_segment(const NmsSegment& seg, const NmsConfig& cfg, int32_t* __restrict__ out_pos,
                                      unsigned char* smem_raw, const NmsPre* pre = nullptr, BoxLoad load_box = BoxLoad()) {
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const int mode = BoxLoad::kMode >= 0 ? BoxLoad::kMode : cfg.mode;
  const float thr = cfg.iou_thr;

  unsigned long long* sK = reinterpret_cast<unsigned long long*>(smem_raw);  // [NMS_WINDOW]
  unsigned long long* sS = sK + NMS_WINDOW;                                  // [NMS_SAMPLES]
  uint32_t* sPos = reinterpret_cast<uint32_t*>(sS + NMS_SAMPLES);            // [NMS_WINDOW]
  float* cC0 = reinterpret_cast<float*>(sPos + NMS_WINDOW);
  float* cC1 = cC0 + NMS_CHUNK;
  float* cC2 = cC1 + NMS_CHUNK;
  float* cC3 = cC2 + NMS_CHUNK;
  float* cAr = cC3 + NMS_CHUNK;
  float* cAt = cAr + NMS_CHUNK;
  int* cCl = reinterpret_cast<int*>(cAt + NMS_CHUNK);
  int* sHead = reinterpret_cast<int*>(cCl + NMS_CHUNK);  // [256] newest kept index per class bucket (-1 = empty)
  float* kC0 = reinterpret_cast<float*>(sHead + 256);
  float* kC1 = kC0 + cfg.max_out;
  float* kC2 = kC1 + cfg.max_out;
  float* kC3 = kC2 + cfg.max_out;
  float* kAr = kC3 + cfg.max_out;
  float* kAt = kAr + cfg.max_out;
  int* kCl = reinterpret_cast<int*>(kAt + cfg.max_out);
  int* kNext = kCl + cfg.max_out;  // per-class chain: previous kept index in the same bucket
  uintptr_t misc_addr = (reinterpret_cast<uintptr_t>(kNext + cfg.max_out) + 15) & ~uintptr_t(15);
  unsigned long long* sMask = reinterpret_cast<unsigned long long*>(misc_addr);  // [64]
  uint32_t* sSupp = reinterpret_cast<uint32_t*>(sMask + 64);                    // [32]
  unsigned long long* sKeptMask = reinterpret_cast<unsigned long long*>(sSupp + 32);
  int* sScalar = reinterpret_cast<int*>(sKeptMask + 1);  // [0]=gathered [1]=eligible [2]=nk [3]=cut bucket

  if (tid < 256) sHead[tid] = -1;
  const int n = seg.n;
  // window size goal: enough candidates to emit max_out boxes when little is suppressed, small enough that the
  // bitonic sort of the window (the dominant cost of a lightly suppressed image) stays cheap
  const int target = nms_window_target(cfg.max_out, n);
  const int min_win = target >> 1;
  int n_kept = 0;
  unsigned long long klo = 0ull;  // inclusive lower bound of not-yet-consumed keys
  bool exhausted = (n <= 0);

  int* sBins = reinterpret_cast<int*>(sS);                    // [2 * NMS_BINS]: bucket counts / starts, chain heads
  unsigned short* sOrd = reinterpret_cast<unsigned short*>(sS);  // [NMS_WINDOW] order of the window (aliases the counts)
  int* sNext = reinterpret_cast<int*>(cC0);                    // [NMS_WINDOW] bucket chains (the candidate tile is idle then)
  uint32_t* sRed = reinterpret_cast<uint32_t*>(sMask);        // 96 words of reduction scratch (64 x 8 bytes available)
  while (!exhausted && n_kept < cfg.max_out) {
    // ---------------- 1. choose and gather the window [klo, khi) ----------------
    unsigned long long khi = ~0ull;   // exclusive upper bound; ~0 = everything that is left
    int n_win = 0;
    bool gathered = false, fallback = false, sorted_in_place = false;
    // Source of the selection passes: the whole segment, or — first window of a large segment — the list that several
    // CTAs pre-gathered below a sampled pivot (all eligible keys < *pre->khi: a superset of the true top of the segment,
    // whose size varies with the sample; up to NMS_PRE_CAP keys, so a generous pivot never overflows).
    bool use_pre = false;
    int src_n = n;
    if (pre && klo == 0ull) {
      const int c = *pre->count, e = *pre->eligible;
      if (e == 0) { exhausted = true; break; }
      if (c >= 1 && c <= NMS_PRE_CAP) { use_pre = true; src_n = c; }
    }
    // one sweep over the source: body(i, K) for every eligible key that is left; NMS_LOADS independent loads in flight per
    // thread (a plain strided loop serialises on the L2 latency: 48 dependent round trips per pass at 49 k candidates)
    // A segment of at most NMS_KC keys per thread is read ONCE: the keys stay in registers for the range, histogram and
    // gather passes (three L2 / L1 round trips per pass otherwise — at 5 k candidates the passes are pure latency).
    const bool small_seg = BoxLoad::kKeyCache && !use_pre && src_n <= NMS_KC * THREADS;
    unsigned long long Kc[NMS_KC];
    uint32_t kc_ok = 0u;
    if (small_seg) {
      float sv[NMS_KC];
      uint32_t ov[NMS_KC];
#pragma unroll
      for (int u = 0; u < NMS_KC; ++u) {
        const int i = tid + u * THREADS;
        sv[u] = (i < src_n) ? seg.scores[i] : 0.0f;
        ov[u] = (i < src_n && seg.order_id) ? seg.order_id[i] : (uint32_t)i;
      }
#pragma unroll
      for (int u = 0; u < NMS_KC; ++u) {
        const int i = tid + u * THREADS;
        Kc[u] = ((unsigned long long)nms_dkey(sv[u]) << 32) | ov[u];
        if ((i < src_n) && !(cfg.use_score_thr && (sv[u] < cfg.score_thr)) && (Kc[u] >= klo)) kc_ok |= 1u << u;
      }
    }
    auto for_each_key = [&](auto&& body) {
      if (small_seg) {
#pragma unroll
        for (int u = 0; u < NMS_KC; ++u) if ((kc_ok >> u) & 1u) body(tid + u * THREADS, Kc[u]);
        return;
      }
      for (int i0 = tid; i0 < src_n; i0 += NMS_LOADS * THREADS) {
        unsigned long long K[NMS_LOADS];
        bool ok[NMS_LOADS];
        if (use_pre) {
#pragma unroll
          for (int u = 0; u < NMS_LOADS; ++u) {
            const int i = i0 + u * THREADS;
            ok[u] = i < src_n;
            K[u] = ok[u] ? pre->keys[i] : 0ull;
          }
        } else {
          float sv[NMS_LOADS];
          uint32_t ov[NMS_LOADS];
#pragma unroll
          for (int u = 0; u < NMS_LOADS; ++u) {
            const int i = i0 + u * THREADS;
            sv[u] = (i < src_n) ? seg.scores[i] : 0.0f;
            ov[u] = (i < src_n && seg.order_id) ? seg.order_id[i] : (uint32_t)i;
          }
#pragma unroll
          for (int u = 0; u < NMS_LOADS; ++u) {
            const int i = i0 + u * THREADS;
            K[u] = ((unsigned long long)nms_dkey(sv[u]) << 32) | ov[u];
            ok[u] = (i < src_n) && !(cfg.use_score_thr && (sv[u] < cfg.score_thr)) && (K[u] >= klo);
          }
        }
#pragma unroll
        for (int u = 0; u < NMS_LOADS; ++u) if (ok[u]) body(i0 + u * THREADS, K[u]);
      }
    };
    bool win_range = false;           // range of the gathered window's keys, known from the selection passes
    uint32_t win_mn = 0u, win_mx = 0u;
    {
      // G1: range and number of the eligible keys that are left.  A large source is only SAMPLED for its range (one key per
      // thread): the buckets stay monotone whatever the bounds are (nms_bin clamps), so the cut below is still exact — keys
      // better than the best sample merely share bucket 0 — and the count comes out of the histogram pass.  One full pass
      // over the scores less (12 of the 35 us the three passes cost at 49 k candidates).
      uint32_t dmin = 0xffffffffu, dmax = 0u;
      int n_el = 0;
      bool sampled = BoxLoad::kSampleRange && !small_seg && src_n > 2 * NMS_WINDOW;
      if (sampled) {
        const int i = (int)(((long long)tid * src_n) / THREADS);
        unsigned long long K;
        bool ok;
        if (use_pre) { K = pre->keys[i]; ok = true; }
        else {
          const float sv = seg.scores[i];
          K = ((unsigned long long)nms_dkey(sv) << 32) | (seg.order_id ? seg.order_id[i] : (uint32_t)i);
          ok = !(cfg.use_score_thr && (sv < cfg.score_thr)) && (K >= klo);
        }
        if (ok) { n_el = 1; dmin = dmax = (uint32_t)(K >> 32); }
        nms_block_minmaxsum<THREADS>(dmin, dmax, n_el, sRed);
        if (n_el < 16) { sampled = false; dmin = 0xffffffffu; dmax = 0u; n_el = 0; }   // too few eligible samples: count properly
      }
      if (!sampled) {
        for_each_key([&](int, unsigned long long K) {
          const uint32_t d = (uint32_t)(K >> 32);
          ++n_el; dmin = min(dmin, d); dmax = max(dmax, d);
        });
        nms_block_minmaxsum<THREADS>(dmin, dmax, n_el, sRed);
        if (n_el == 0) { exhausted = true; break; }
      }
      const float scale = nms_bin_scale(dmin, dmax);
      int cut = NMS_BINS - 1;
      if (sampled || n_el > NMS_WINDOW) {
        // G2: histogram of the buckets; G3: the bucket where the cumulative count reaches the target
        for (int b = tid; b < NMS_BINS; b += THREADS) sBins[b] = 0;
        __syncthreads();
        for_each_key([&](int, unsigned long long K) { atomicAdd(&sBins[nms_bin((uint32_t)(K >> 32), dmin, scale)], 1); });
        __syncthreads();
        const int total = nms_block_scan_bins<THREADS>(sBins, sRed, target, &sScalar[3]);
        if (sampled) n_el = total;      // (>= 16: the samples are among them)
        cut = sScalar[3];
        const int upto = (cut + 1 < NMS_BINS) ? sBins[cut + 1] : n_el;   // keys in buckets 0..cut
        fallback = upto > NMS_WINDOW;   // one bucket alone overflows the window (masses of near-equal scores)
        __syncthreads();
        if (fallback && use_pre) {      // cannot happen short of thousands of tied scores: redo on the whole segment
          use_pre = false; src_n = n; fallback = true;
        }
      }
      if (!fallback) {
        // G4: gather buckets 0..cut (unordered)
        if (tid == 0) sScalar[0] = 0;
        __syncthreads();
        for_each_key([&](int i, unsigned long long K) {
          if (nms_bin((uint32_t)(K >> 32), dmin, scale) > cut) return;
          const uint32_t grp = __activemask();   // one atomic per group of lanes that arrive together
          const int leader = __ffs(grp) - 1;
          int slot = 0;
          if (lane == leader) slot = atomicAdd(&sScalar[0], __popc(grp));
          slot = __shfl_sync(grp, slot, leader) + __popc(grp & ((1u << lane) - 1u));
          sK[slot] = K; sPos[slot] = use_pre ? pre->pos[i] : (uint32_t)i;
        });
        __syncthreads();
        n_win = sScalar[0];
        gathered = true;
        win_range = !sampled; win_mn = dmin; win_mx = dmax;   // (a sampled range would pile the best keys into one ordering bucket)
        if (cut < NMS_BINS - 1) {       // keys of buckets 0..cut lie below dmin + (cut + 1) / scale (an estimate is enough)
          const float lim = (float)(cut + 1) / scale;
          if (lim < (float)(dmax - dmin)) win_mx = dmin + (uint32_t)lim + 1u;
        }
        // the window holds everything that is left only if nothing was cut here AND the pre-gathered list was complete
        const bool complete = (n_win >= n_el) && (!use_pre || *pre->count >= *pre->eligible);
        if (!complete) khi = 1ull;   // placeholder: the real bound (largest key of the window + 1) is set after ordering
        __syncthreads();
      }
    }
    if (!gathered) {
      // fallback of round 1: pivot from sorted samples, rescale / bisect until the window fits, bitonic sort
      const bool take_all = (n <= NMS_WINDOW);
      unsigned long long rank = 0;
      int n_samp = 256;  // enough samples for a pivot rank of >= ~48 (relative spread of the admitted count <= ~15 %)
      while (n_samp < NMS_SAMPLES && (long long)n_samp * target < 48ll * n) n_samp <<= 1;
      khi = ~0ull;
      if (!take_all) {
        for (int t = tid; t < n_samp; t += THREADS) {
          const int i = (int)(((long long)t * n) / n_samp);
          const float s = seg.scores[i];
          const uint32_t oid = seg.order_id ? seg.order_id[i] : (uint32_t)i;
          const unsigned long long K = ((unsigned long long)nms_dkey(s) << 32) | oid;
          const bool el = !(cfg.use_score_thr && (s < cfg.score_thr)) && (K >= klo);
          sS[t] = el ? K : ~0ull;
        }
        __syncthreads();
        nms_bitonic<THREADS>(sS, nullptr, n_samp);
        rank = ((unsigned long long)target * (unsigned long long)n_samp) / (unsigned long long)n;
        if (rank < 2ull) rank = 2ull;
        khi = rank >= (unsigned long long)n_samp ? ~0ull : sS[rank];
      }
      unsigned long long b_lo = klo, b_hi = ~0ull;  // bisection bounds: khi <= b_lo admits too few, khi >= b_hi too many
      for (int attempt = 0; attempt < 80; ++attempt) {
        if (tid == 0) { sScalar[0] = 0; sScalar[1] = 0; }
        __syncthreads();
        int my_el = 0;
        for (int i = tid; i < n; i += THREADS) {
          const float s = seg.scores[i];
          if (cfg.use_score_thr && (s < cfg.score_thr)) continue;
          const uint32_t oid = seg.order_id ? seg.order_id[i] : (uint32_t)i;
          const unsigned long long K = ((unsigned long long)nms_dkey(s) << 32) | oid;
          if (K < klo) continue;
          ++my_el;
          if (khi == ~0ull || K < khi) {
            const int slot = atomicAdd(&sScalar[0], 1);
            if (slot < NMS_WINDOW) { sK[slot] = K; sPos[slot] = (uint32_t)i; }
          }
        }
        my_el = warp_sum_i(my_el);
        if (lane == 0 && my_el) atomicAdd(&sScalar[1], my_el);
        __syncthreads();
        const int c = sScalar[0], e = sScalar[1];
        __syncthreads();
        if (e == 0) { n_win = 0; break; }
        const bool too_many = c > NMS_WINDOW;
        const bool too_few = (c < min_win) && (c < e);
        if (!too_many && !too_few) {
          n_win = c;
          if (c >= e) khi = ~0ull;  // the window holds everything that was left
          break;
        }
        // adjust the pivot: rescale the sample rank first, then bisect on the key value
        if (too_many) b_hi = khi; else b_lo = khi;
        unsigned long long next = 0ull;
        bool have = false;
        if (attempt < 3 && !take_all) {
          unsigned long long r2 = c > 0 ? (rank * (unsigned long long)target) / (unsigned long long)c : rank * 8ull;
          if (too_few && r2 <= rank) r2 = rank + 1ull;
          if (too_many && r2 >= rank) r2 = rank > 0ull ? rank - 1ull : 0ull;
          rank = r2;
          next = rank >= (unsigned long long)n_samp ? ~0ull : sS[rank];
          have = (next > b_lo) && (next < b_hi || b_hi == ~0ull) && (next != khi);
        }
        if (!have) next = b_lo + ((b_hi - b_lo) >> 1);
        if (next == khi || next <= b_lo) next = b_lo + 1ull;  // keys are unique: a one-key step cannot skip the band
        khi = next;
      }
      sorted_in_place = n_win > 0;
    }
    if (n_win == 0) { exhausted = true; break; }
    if (sorted_in_place) {
      int npad = 64;
      while (npad < n_win) npad <<= 1;
      for (int t = tid; t < npad; t += THREADS)
        if (t >= n_win) { sK[t] = ~0ull; sPos[t] = 0xffffffffu; }
      __syncthreads();
      nms_bitonic<THREADS>(sK, sPos, npad);
      for (int t = tid; t < n_win; t += THREADS) sOrd[t] = (unsigned short)t;
      __syncthreads();
    } else {
      nms_bucket_order<THREADS>(sK, n_win, sBins, sNext, sRed, sOrd, win_range, win_mn, win_mx);
      if (khi == 1ull) khi = sK[sOrd[n_win - 1]] + 1ull;   // everything not gathered has a larger key (bucket > cut)
    }

    // ---------------- 2. consume the window in tiles of 64 sorted candidates, lazily ----------------
    // Only as many tiles as are needed to emit max_out boxes are ever touched: a tile is first tested against
    // every box emitted so far (64 x n_kept pairs spread over the 1024 threads), then resolved internally with a
    // 64x64 ballot bitmask and a one-warp sweep.  Work is O(emitted^2), independent of the window size.
    for (int w0 = 0; w0 < n_win && n_kept < cfg.max_out; w0 += NMS_CHUNK) {
      const int n_chunk = min(NMS_CHUNK, n_win - w0);
      for (int ct = tid; ct < n_chunk; ct += THREADS) {
        const uint32_t p = sPos[sOrd[w0 + ct]];
        const float4 b = load_box(seg, p);
        const BoxT mine = bm_prep(b.x, b.y, b.z, b.w, METRIC);
        cC0[ct] = mine.c0; cC1[ct] = mine.c1; cC2[ct] = mine.c2; cC3[ct] = mine.c3;
        cAr[ct] = mine.area; cAt[ct] = mine.at; cCl[ct] = seg.classes ? seg.classes[p] : 0;
      }
      if (tid < 2) sSupp[tid] = 0u;
      __syncthreads();
      if (mode == B200_NMS_BY_CLASS) {
        // ---- per-class NMS: classes never interact, so the chunk is split by class bucket and every bucket is resolved
        // by its own warp (greedy in rank order inside the bucket); the survivors are then emitted in global rank order.
        // Exact: a candidate is dropped iff an EMITTED better-ranked box of its class suppresses it, and every surviving
        // better-ranked box inside the cap is emitted.  No tile loop: ~8 CTA barriers per 1024 candidates.
        unsigned short* sTab = reinterpret_cast<unsigned short*>(sK);          // [32 blocks][256 buckets] counts -> offsets
        unsigned short* sMem = sTab + 32 * 256;                                 // [NMS_CHUNK] members, bucket-major, rank order
        int* sBase = reinterpret_cast<int*>(sMem + NMS_CHUNK);                  // [257] bucket starts
        unsigned char* sAlive = reinterpret_cast<unsigned char*>(sBase + 260);  // [NMS_CHUNK] not suppressed by an earlier chunk / window
        unsigned long long* sSet = reinterpret_cast<unsigned long long*>(sAlive + NMS_CHUNK);  // [256] per bucket: alive members (bit = position)
        int* sPB = reinterpret_cast<int*>(sSet + 256);                           // [257] pair-index starts of the buckets
        unsigned short* sQ = reinterpret_cast<unsigned short*>(sPB + 260);       // [NMS_CHUNK] candidate -> its slot in sMem
        unsigned long long* sBy = sS + NMS_SAMPLES / 2;   // [NMS_CHUNK] per member: which better-ranked bucket mates suppress it (sOrd holds the first half of sS)
        static_assert(32 * 256 * 2 + NMS_CHUNK * 2 + 260 * 4 + NMS_CHUNK + 256 * 8 + 260 * 4 + NMS_CHUNK * 2 <= NMS_WINDOW * 8, "per-class scratch exceeds the key window");
        static_assert(NMS_WINDOW * 2 <= NMS_SAMPLES * 4 && NMS_CHUNK * 8 <= NMS_SAMPLES * 4, "sOrd / sBy do not fit the sample array");
        constexpr int NW = THREADS / 32;
        constexpr int BUCKET_MAX = 64;   // buckets up to this size are resolved from suppression words, larger ones by the warp loop
        // (1) against the boxes kept by earlier chunks / windows; clear the count table and the suppression words
        for (int ct = tid; ct < n_chunk; ct += THREADS) {
          bool supp = false;
          if (n_kept > 0) {
            const int ccls = cCl[ct];
            BoxT cb; cb.c0 = cC0[ct]; cb.c1 = cC1[ct]; cb.c2 = cC2[ct]; cb.c3 = cC3[ct]; cb.area = cAr[ct]; cb.at = cAt[ct];
            for (int k = sHead[(uint32_t)ccls & 255u]; k >= 0; k = kNext[k]) {
              if (kCl[k] != ccls) continue;
              BoxT kb; kb.c0 = kC0[k]; kb.c1 = kC1[k]; kb.c2 = kC2[k]; kb.c3 = kC3[k]; kb.area = kAr[k]; kb.at = kAt[k];
              if (nms_suppresses<METRIC>(kb, ccls, cb, ccls, mode, thr)) { supp = true; break; }
            }
          }
          sAlive[ct] = supp ? 0 : 1;
          sBy[ct] = 0ull;
        }
        for (int i = tid; i < 32 * 256 / 2; i += THREADS) reinterpret_cast<uint32_t*>(sTab)[i] = 0u;
        for (int i = tid; i < 256; i += THREADS) sSet[i] = 0ull;
        __syncthreads();
        // (2) stable split by bucket: 32-candidate blocks in rank order; intra-block rank by match_any, block counts in sTab
        const int n_blk = (n_chunk + 31) >> 5;
        for (int blk = warp; blk < n_blk; blk += NW) {
          const int ct = (blk << 5) + lane;
          const uint32_t bucket = ct < n_chunk ? ((uint32_t)cCl[ct] & 255u) : 0xffffu;
          const uint32_t peers = __match_any_sync(0xffffffffu, bucket);
          if (ct < n_chunk && (peers & ((1u << lane) - 1u)) == 0u) sTab[blk * 256 + bucket] = (unsigned short)__popc(peers);
        }
        __syncthreads();
        for (int b = tid; b < 256; b += THREADS) {   // per bucket: exclusive prefix over the blocks, total into sBase[b + 1]
          int t[NMS_CHUNK / 32], run = 0;              // all counts are loaded before the first store (independent loads)
#pragma unroll
          for (int blk = 0; blk < NMS_CHUNK / 32; ++blk) t[blk] = (blk < n_blk) ? (int)sTab[blk * 256 + b] : 0;
#pragma unroll
          for (int blk = 0; blk < NMS_CHUNK / 32; ++blk) { if (blk < n_blk) sTab[blk * 256 + b] = (unsigned short)run; run += t[blk]; }
          sBase[b + 1] = run;
        }
        __syncthreads();
        if (warp == 0) {   // bucket starts: exclusive prefix of the 256 totals; pair-index starts: the same over m (m - 1) / 2
          int v[8], pv[8], local = 0, plocal = 0;
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            v[k] = sBase[lane * 8 + k + 1]; local += v[k];
            pv[k] = (v[k] <= BUCKET_MAX) ? (v[k] * (v[k] - 1)) >> 1 : 0; plocal += pv[k];
          }
          int incl = local, pincl = plocal;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o), pt = __shfl_up_sync(0xffffffffu, pincl, o);
            if (lane >= o) { incl += t; pincl += pt; }
          }
          int run = incl - local, prun = pincl - plocal;
          __syncwarp();
#pragma unroll
          for (int k = 0; k < 8; ++k) { sBase[lane * 8 + k] = run; run += v[k]; sPB[lane * 8 + k] = prun; prun += pv[k]; }
          if (lane == 31) { sBase[256] = run; sPB[256] = prun; }
        }
        __syncthreads();
        for (int blk = warp; blk < n_blk; blk += NW) {
          const int ct = (blk << 5) + lane;
          const uint32_t bucket = ct < n_chunk ? ((uint32_t)cCl[ct] & 255u) : 0xffffu;
          const uint32_t peers = __match_any_sync(0xffffffffu, bucket);
          if (ct < n_chunk) {
            const int base = sBase[bucket];
            const int pos = sTab[blk * 256 + bucket] + __popc(peers & ((1u << lane) - 1u));
            sMem[base + pos] = (unsigned short)ct;
            sQ[ct] = (unsigned short)(base + pos);
            if (sAlive[ct] && pos < BUCKET_MAX) atomicOr(&sSet[bucket], 1ull << pos);   // (only read for buckets <= BUCKET_MAX)
          }
        }
        __syncthreads();
        // (3) inside a bucket.  The pairs (i < j) of all buckets form one flat index space (bucket starts in sPB, a triangle
        // inside a bucket): every thread tests an equal share of them and ORs bit i into member j's word when i (same class)
        // suppresses j.  Then one thread per bucket walks its members in rank order with the alive set in a register: member
        // t stays iff it was alive and no ALIVE better-ranked mate suppresses it — the greedy recurrence itself, ~5 dependent
        // ALU steps per member.  (A warp per bucket walking shared-memory state took 14 us of the 36 us of a 416x416 image —
        // 10 members per class, three buckets per warp, the slowest warp decides; a thread per member 5 us.)
        {
          const int P = sPB[256];
          const int per = (P + THREADS - 1) / THREADS;
          int e = tid * per;
          const int e_end = min(P, e + per);
          if (e < e_end) {
            int lo = 0, hi = 256;                          // sPB[lo] <= e < sPB[hi]
            while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (sPB[mid] <= e) lo = mid; else hi = mid; }
            int bkt = lo, base = sBase[bkt], m = sBase[bkt + 1] - base;
            const int r = e - sPB[bkt];
            int j = (int)((1.0f + sqrtf(1.0f + 8.0f * (float)r)) * 0.5f);
            while ((j * (j - 1)) >> 1 > r) --j;
            while (((j + 1) * j) >> 1 <= r) ++j;
            int i = r - ((j * (j - 1)) >> 1);
            int cj = sMem[base + j];
            BoxT bj; bj.c0 = cC0[cj]; bj.c1 = cC1[cj]; bj.c2 = cC2[cj]; bj.c3 = cC3[cj]; bj.area = cAr[cj]; bj.at = cAt[cj];
            int cls_j = cCl[cj];
            for (;;) {
              const int ci = sMem[base + i];
              if (cCl[ci] == cls_j) {                      // classes sharing a bucket (ids 256 apart) do not interact
                BoxT bi; bi.c0 = cC0[ci]; bi.c1 = cC1[ci]; bi.c2 = cC2[ci]; bi.c3 = cC3[ci]; bi.area = cAr[ci]; bi.at = cAt[ci];
                if (nms_suppresses<METRIC>(bi, cls_j, bj, cls_j, mode, thr)) atomicOr(&sBy[base + j], 1ull << i);
              }
              if (++e >= e_end) break;
              if (++i == j) {
                i = 0;
                if (++j == m) {                            // next bucket that has pairs (exists: e < P)
                  do { ++bkt; base = sBase[bkt]; m = sBase[bkt + 1] - base; } while (m < 2 || m > BUCKET_MAX);
                  j = 1;
                }
                cj = sMem[base + j];
                bj.c0 = cC0[cj]; bj.c1 = cC1[cj]; bj.c2 = cC2[cj]; bj.c3 = cC3[cj]; bj.area = cAr[cj]; bj.at = cAt[cj];
                cls_j = cCl[cj];
              }
            }
          }
        }
        __syncthreads();
        // (buckets spread over all warps: a warp waits for the largest of its buckets)
        for (int b = tid / (THREADS / 256); b < 256 && tid % (THREADS / 256) == 0; b += 256) {
          const int base = sBase[b], m = sBase[b + 1] - base;
          if (m < 2 || m > BUCKET_MAX) continue;
          const unsigned long long a0 = sSet[b];
          unsigned long long alive = 0ull;
#pragma unroll 4
          for (int t = 0; t < m; ++t) {
            const bool a = ((a0 >> t) & 1ull) && !(sBy[base + t] & alive);
            alive |= (unsigned long long)a << t;
          }
          sSet[b] = alive;
        }
        for (int b = warp; b < 256; b += NW) {   // oversized buckets: a warp per bucket, greedy in rank order, state in sAlive
          const int base = sBase[b], m = sBase[b + 1] - base;
          if (m <= BUCKET_MAX) continue;                 // warp-uniform
          for (int i = 0; i + 1 < m; ++i) {
            const int ci = sMem[base + i];
            if (!sAlive[ci]) continue;                   // warp-uniform
            BoxT bi; bi.c0 = cC0[ci]; bi.c1 = cC1[ci]; bi.c2 = cC2[ci]; bi.c3 = cC3[ci]; bi.area = cAr[ci]; bi.at = cAt[ci];
            const int cls_i = cCl[ci];
            for (int j = i + 1 + lane; j < m; j += 32) {
              const int cj = sMem[base + j];
              if (!sAlive[cj] || cCl[cj] != cls_i) continue;
              BoxT bj; bj.c0 = cC0[cj]; bj.c1 = cC1[cj]; bj.c2 = cC2[cj]; bj.c3 = cC3[cj]; bj.area = cAr[cj]; bj.at = cAt[cj];
              if (nms_suppresses<METRIC>(bi, cls_i, bj, cls_i, mode, thr)) sAlive[cj] = 0;
            }
            __syncwarp();
          }
        }
        __syncthreads();
        // (4) emit the survivors in rank order, up to the cap
        for (int c0 = 0; c0 < n_chunk && n_kept < cfg.max_out; c0 += THREADS) {
          const int ct = c0 + tid;
          bool a = false;
          if (ct < n_chunk) {
            const uint32_t bucket = (uint32_t)cCl[ct] & 255u;
            const int base = sBase[bucket];
            a = (sBase[bucket + 1] - base <= BUCKET_MAX) ? ((sSet[bucket] >> ((int)sQ[ct] - base)) & 1ull) != 0ull : sAlive[ct] != 0;
          }
          const uint32_t bal = __ballot_sync(0xffffffffu, a);
          if (lane == 0) sRed[warp] = (uint32_t)__popc(bal);
          __syncthreads();
          int before = 0, total = 0;
#pragma unroll
          for (int w = 0; w < NW; ++w) { const int t = (int)sRed[w]; if (w < warp) before += t; total += t; }
          const int slot = n_kept + before + __popc(bal & ((1u << lane) - 1u));
          if (a && slot < cfg.max_out) {
            kC0[slot] = cC0[ct]; kC1[slot] = cC1[ct]; kC2[slot] = cC2[ct]; kC3[slot] = cC3[ct];
            kAr[slot] = cAr[ct]; kAt[slot] = cAt[ct]; kCl[slot] = cCl[ct];
            out_pos[slot] = (int32_t)sPos[sOrd[w0 + ct]];
            kNext[slot] = atomicExch(&sHead[(uint32_t)cCl[ct] & 255u], slot);
          }
          n_kept = min(cfg.max_out, n_kept + total);
          __syncthreads();
        }
        continue;
      }
      const int n_tiles = (n_chunk + 63) >> 6;
      for (int T = 0; T < n_tiles && n_kept < cfg.max_out; ++T) {
        const int t0 = T << 6;
        // phase 1: tile candidates vs the kept list.  warp w: candidates 32*(w&1)..+31, kept indices (w>>1) + (THREADS/64) j
        {
          const int c = ((warp & 1) << 5) + lane;
          const int gj = t0 + c;
          bool supp = false;
          if (gj < n_chunk && n_kept > 0) {
            BoxT cb; cb.c0 = cC0[gj]; cb.c1 = cC1[gj]; cb.c2 = cC2[gj]; cb.c3 = cC3[gj]; cb.area = cAr[gj]; cb.at = cAt[gj];
            const int ccls = cCl[gj];
            if (mode == B200_NMS_BY_CLASS) {
              // only emitted boxes of the same class can suppress: walk the class bucket's chain (two warps)
              if (warp < 2) {
                for (int k = sHead[(uint32_t)ccls & 255u]; k >= 0; k = kNext[k]) {
                  if (kCl[k] != ccls) continue;
                  BoxT kb; kb.c0 = kC0[k]; kb.c1 = kC1[k]; kb.c2 = kC2[k]; kb.c3 = kC3[k]; kb.area = kAr[k]; kb.at = kAt[k];
                  if (nms_suppresses<METRIC>(kb, ccls, cb, ccls, mode, thr)) { supp = true; break; }
                }
              }
            } else {
              for (int k = warp >> 1; k < n_kept; k += THREADS / 64) {
                BoxT kb; kb.c0 = kC0[k]; kb.c1 = kC1[k]; kb.c2 = kC2[k]; kb.c3 = kC3[k]; kb.area = kAr[k]; kb.at = kAt[k];
                if (nms_suppresses<METRIC>(kb, 0, cb, 0, mode, thr)) { supp = true; break; }
              }
            }
          }
          const uint32_t bits = __ballot_sync(0xffffffffu, supp);
          if (lane == 0 && bits) atomicOr(&sSupp[warp & 1], bits);  // sSupp: bits of tile candidates suppressed by the kept list
        }
        __syncthreads();
        unsigned long long tile_alive = ~((unsigned long long)sSupp[0] | ((unsigned long long)sSupp[1] << 32));
        if (n_chunk - t0 < 64) tile_alive &= (1ull << (n_chunk - t0)) - 1ull;
        // phase 2: intra-tile mask via ballots: warp w owns rows (2048/THREADS) w ... (2 rows at 1024 threads)
#pragma unroll
        for (int rr = 0; rr < 2048 / THREADS; ++rr) {
          const int r = (2048 / THREADS) * warp + rr;
          const int gi = t0 + r;
          const bool row_on = (gi < n_chunk) && ((tile_alive >> r) & 1ull);
          BoxT rb; int rcls = 0;
          rb.c0 = rb.c1 = rb.c2 = rb.c3 = rb.area = rb.at = 0.f;
          if (row_on) { rb.c0 = cC0[gi]; rb.c1 = cC1[gi]; rb.c2 = cC2[gi]; rb.c3 = cC3[gi]; rb.area = cAr[gi]; rb.at = cAt[gi]; rcls = cCl[gi]; }
          uint32_t bits[2];
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const int c = half * 32 + lane;
            const int gj = t0 + c;
            bool pred = false;
            if (row_on && c > r && gj < n_chunk && ((tile_alive >> c) & 1ull)) {
              const int ccls = cCl[gj];
              if (mode != B200_NMS_BY_CLASS || ccls == rcls) {
                BoxT cb; cb.c0 = cC0[gj]; cb.c1 = cC1[gj]; cb.c2 = cC2[gj]; cb.c3 = cC3[gj]; cb.area = cAr[gj]; cb.at = cAt[gj];
                pred = nms_suppresses<METRIC>(rb, rcls, cb, ccls, mode, thr);
              }
            }
            bits[half] = __ballot_sync(0xffffffffu, pred);
          }
          if (lane == 0) sMask[r] = (unsigned long long)bits[0] | ((unsigned long long)bits[1] << 32);
        }
        __syncthreads();
        // one-warp sweep.  lane <-> columns lane and lane + 32: the warp first transposes the 64 x 64 bit matrix (64 broadcast
        // reads; by = the better-ranked rows that suppress the column), then iterates  kept' = alive & ~any(by & kept)  from
        // kept = alive until nothing changes.  The greedy solution is the unique fixed point and position j is final after
        // j + 1 rounds at the latest — in practice after the length of the longest suppression chain (2-4 rounds), where a
        // single thread walking the kept rows paid one dependent shared-memory read per emitted box (1.8 us per tile).
        if (warp == 0) {
          const unsigned long long m0 = ((tile_alive >> lane) & 1ull) ? (sMask[lane] & tile_alive) : 0ull;
          const unsigned long long m1 = ((tile_alive >> (lane + 32)) & 1ull) ? (sMask[lane + 32] & tile_alive) : 0ull;
          const bool any = __any_sync(0xffffffffu, (m0 | m1) != 0ull);
          unsigned long long keptmask = tile_alive;
          const int room = cfg.max_out - n_kept;
          if (any) {
            uint32_t by0_lo = 0u, by0_hi = 0u, by1_lo = 0u, by1_hi = 0u;
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const unsigned long long ra = sMask[i], rb = sMask[i + 32];   // rows of dead candidates are all zero (phase 2)
              by0_lo |= (((uint32_t)ra >> lane) & 1u) << i;
              by1_lo |= (((uint32_t)(ra >> 32) >> lane) & 1u) << i;
              by0_hi |= (((uint32_t)rb >> lane) & 1u) << i;
              by1_hi |= (((uint32_t)(rb >> 32) >> lane) & 1u) << i;
            }
            const unsigned long long by0 = ((unsigned long long)by0_hi << 32) | by0_lo, by1 = ((unsigned long long)by1_hi << 32) | by1_lo;
            const bool a0 = (tile_alive >> lane) & 1ull, a1 = (tile_alive >> (lane + 32)) & 1ull;
            for (;;) {
              const uint32_t k0 = __ballot_sync(0xffffffffu, a0 && !(by0 & keptmask));
              const uint32_t k1 = __ballot_sync(0xffffffffu, a1 && !(by1 & keptmask));
              const unsigned long long next = ((unsigned long long)k1 << 32) | k0;
              if (next == keptmask) break;
              keptmask = next;
            }
          }
          if (lane == 0) {
            int nk = __popcll(keptmask);
            while (nk > room) {  // keep only the first `room` of them
              const int hi = 63 - __clzll((long long)keptmask);
              keptmask &= ~(1ull << hi);
              --nk;
            }
            *sKeptMask = keptmask;
            sScalar[2] = __popcll(keptmask);
            sSupp[0] = 0u; sSupp[1] = 0u;  // reset the suppressed bits for the next tile
          }
        }
        __syncthreads();
        const unsigned long long keptmask = *sKeptMask;
        const int nk = sScalar[2];
        // emit: append to the kept list
        if (tid < 64 && ((keptmask >> tid) & 1ull)) {
          const int gi = t0 + tid;
          const int slot = n_kept + __popcll(keptmask & ((1ull << tid) - 1ull));
          kC0[slot] = cC0[gi]; kC1[slot] = cC1[gi]; kC2[slot] = cC2[gi]; kC3[slot] = cC3[gi];
          kAr[slot] = cAr[gi]; kAt[slot] = cAt[gi]; kCl[slot] = cCl[gi];
          out_pos[slot] = (int32_t)sPos[sOrd[w0 + gi]];
          if (mode == B200_NMS_BY_CLASS) kNext[slot] = atomicExch(&sHead[(uint32_t)cCl[gi] & 255u], slot);
        }
        n_kept += nk;
        __syncthreads();
      }
      __syncthreads();
    }
    if (khi == ~0ull) exhausted = true;
    klo = khi;
    __syncthreads();
  }
  return n_kept;
}

// ---- multi-CTA pre-selection of the first window ---------------------------------------------------------
struct NmsPreselectParams {
  const float* scores;          // [num_segments, stride]
  const uint32_t* order_id;     // [num_segments, stride] or nullptr
  const int32_t* counts;        // [num_segments] candidates per segment
  int stride;                   // elements between segments
  int slices;                   // CTAs per segment
  int use_score_thr; float score_thr;
  unsigned long long* keys; uint32_t* pos;  // [num_segments, NMS_PRE_CAP]
  int* count; int* eligible; unsigned long long* khi;  // [num_segments] (count/eligible zeroed by the caller)
};

#define NMS_PRE_SAMPLES 4096
#define NMS_PIVOT_SMEM ((size_t)NMS_PRE_SAMPLES * 8 + 2 * NMS_BINS * 4 + NMS_PRE_SAMPLES * 4 + 512)

// One CTA per segment: pivot = the sample whose rank should admit ~NMS_TARGET candidates (up to 4096 strided samples,
// so the admitted count has a relative spread of ~1/sqrt(rank) and stays inside [1024, 4096] with high probability).
static __device__ void nms_pivot_body(const NmsPreselectParams& p, unsigned char* smem_raw) {
  unsigned long long* sS = reinterpret_cast<unsigned long long*>(smem_raw);  // [NMS_PRE_SAMPLES]
  const int tid = threadIdx.x;
  const int seg = blockIdx.x;
  const int n = p.counts[seg];
  const float* scores = p.scores + (size_t)seg * p.stride;
  const uint32_t* oid_base = p.order_id ? p.order_id + (size_t)seg * p.stride : nullptr;
  unsigned long long khi = ~0ull;
  if (n > NMS_WINDOW) {
    // enough samples for a pivot rank of >= ~32 (relative spread of the admitted count <= ~18 %)
    int ns = 512;
    while (ns < NMS_PRE_SAMPLES && (long long)ns * NMS_TARGET_LARGE < 32ll * n) ns <<= 1;
    for (int t = tid; t < ns; t += NMS_THREADS) {
      const int i = (int)(((long long)t * n) / ns);
      const float s = scores[i];
      const uint32_t oid = oid_base ? oid_base[i] : (uint32_t)i;
      const unsigned long long K = ((unsigned long long)nms_dkey(s) << 32) | oid;
      sS[t] = (p.use_score_thr && (s < p.score_thr)) ? ~0ull : K;
    }
    __syncthreads();
    // rank-th smallest sample by bucket ordering (ineligible samples carry the largest key and sort last; they share
    // one key, so their mutual order is arbitrary, which is harmless: only eligible ranks are ever looked up)
    int* bins = reinterpret_cast<int*>(sS + NMS_PRE_SAMPLES);
    int* nxt = bins + 2 * NMS_BINS;
    uint32_t* red = reinterpret_cast<uint32_t*>(nxt + NMS_PRE_SAMPLES);
    unsigned short* ord = reinterpret_cast<unsigned short*>(bins);
    nms_bucket_order<NMS_THREADS>(sS, ns, bins, nxt, red, ord);
    unsigned long long rank = ((unsigned long long)NMS_TARGET_LARGE * (unsigned long long)ns) / (unsigned long long)n;
    if (rank < 2ull) rank = 2ull;
    khi = rank >= (unsigned long long)ns ? ~0ull : sS[ord[rank]];
  }
  if (tid == 0) p.khi[seg] = khi;
}

// `slices` CTAs per segment: each scans its slice (4 independent loads in flight per thread) and appends the eligible
// keys below the pivot to the segment's window in global memory with warp-aggregated atomics.
#define NMS_PG_STAGE 1024   // selected keys a CTA stages in shared memory before its single append to the segment's list
#define NMS_PG_LOADS 8      // independent loads of each array a thread keeps in flight

static __device__ void nms_pregather_body(const NmsPreselectParams& p) {
  __shared__ unsigned long long s_keys[NMS_PG_STAGE];
  __shared__ uint32_t s_pos[NMS_PG_STAGE];
  __shared__ int s_n, s_el, s_base;
  const int tid = threadIdx.x, lane = tid & 31;
  const int seg = blockIdx.x / p.slices, slice = blockIdx.x - seg * p.slices;
  const int n = p.counts[seg];
  const float* scores = p.scores + (size_t)seg * p.stride;
  const uint32_t* oid_base = p.order_id ? p.order_id + (size_t)seg * p.stride : nullptr;
  const unsigned long long khi = p.khi[seg];
  const int lo = (int)(((long long)slice * n) / p.slices), hi = (int)(((long long)(slice + 1) * n) / p.slices);
  if (tid == 0) { s_n = 0; s_el = 0; }
  __syncthreads();
  int my_el = 0;
  const int T = blockDim.x;
  for (int i0 = lo; i0 < hi; i0 += NMS_PG_LOADS * T) {
    float sv[NMS_PG_LOADS]; uint32_t ov[NMS_PG_LOADS];
#pragma unroll
    for (int u = 0; u < NMS_PG_LOADS; ++u) {
      const int i = i0 + u * T + tid;
      sv[u] = (i < hi) ? scores[i] : 0.0f;
      ov[u] = (i < hi) ? (oid_base ? oid_base[i] : (uint32_t)i) : 0u;
    }
#pragma unroll
    for (int u = 0; u < NMS_PG_LOADS; ++u) {
      const int i = i0 + u * T + tid;
      if (i < hi && !(p.use_score_thr && (sv[u] < p.score_thr))) {
        const unsigned long long K = ((unsigned long long)nms_dkey(sv[u]) << 32) | ov[u];
        ++my_el;
        if ((khi == ~0ull) || (K < khi)) {
          // staged in shared memory (an atomic there returns in a few cycles; a global one per hit stalled the warp for a
          // round trip); the rare overflow goes straight to the list
          const int slot = atomicAdd(&s_n, 1);
          if (slot < NMS_PG_STAGE) { s_keys[slot] = K; s_pos[slot] = (uint32_t)i; }
          else {
            const int g = atomicAdd(&p.count[seg], 1);
            if (g < NMS_PRE_CAP) { p.keys[(size_t)seg * NMS_PRE_CAP + g] = K; p.pos[(size_t)seg * NMS_PRE_CAP + g] = (uint32_t)i; }
          }
        }
      }
    }
  }
  my_el = warp_sum_i(my_el);
  if (lane == 0 && my_el) atomicAdd(&s_el, my_el);
  __syncthreads();
  const int staged = min(s_n, NMS_PG_STAGE);
  if (tid == 0) {
    s_base = staged ? atomicAdd(&p.count[seg], staged) : 0;
    if (s_el) atomicAdd(&p.eligible[seg], s_el);
  }
  __syncthreads();
  for (int t = tid; t < staged; t += T) {
    const int g = s_base + t;
    if (g < NMS_PRE_CAP) { p.keys[(size_t)seg * NMS_PRE_CAP + g] = s_keys[t]; p.pos[(size_t)seg * NMS_PRE_CAP + g] = s_pos[t]; }
  }
}

// ---- candidate store of the fused post-processing (yolo_decode.cu, effdet.cu) --------------------------------------
// A filter kernel appends the candidates of every image to the store; one finalize CTA per image then runs the NMS over its
// image's row and gathers the kept rows.  Image i's candidates are slots [i * n_img, i * n_img + counts[i]) of every
// column, in arbitrary order; bit aidx of the image's row of `bitmap` marks each appended flat anchor index.
struct CandStore {
  float4* box; float* score; int32_t* cls; uint32_t* aidx;  // [n_images, n_img]
  float* conf;                  // [n_images, n_img] (YOLO: the conf logit) or nullptr
  int32_t* counts;              // [n_images]
  uint32_t* bitmap;             // [n_images, bitmap_words], only when sel_idx is wanted (else nullptr)
  int bitmap_words, n_img;
  int32_t* pos;                 // [n_images, max_out] NMS output positions
  // first NMS window from the multi-CTA pre-selection (EfficientDet); nullptr unless an image can exceed NMS_PRE_MIN_N
  unsigned long long* pre_keys; uint32_t* pre_pos;          // [n_images, NMS_PRE_CAP]
  int* pre_count; int* pre_elig; unsigned long long* pre_khi;  // [n_images]
};

// Byte offsets of the store's blocks in a workspace.  Each block is 256-aligned on its own.  counts, the pre-selection
// counters and the bitmap lead, so one memset of zeroed(sel_idx) bytes clears everything that is counted into.
struct CandLayout {
  size_t counts, pre_count, pre_elig, bitmap, box, score, cls, conf, aidx, pos, pre_khi, pre_keys, pre_pos, total;
  int n_img, bitmap_words;
  bool with_conf, with_preselect;
  size_t zeroed(bool sel_idx) const { return sel_idx ? box : bitmap; }
};

static inline CandLayout cand_layout(int n_images, int n_img, int max_out, bool with_conf, bool with_preselect) {
  CandLayout L = {};
  L.n_img = n_img; L.bitmap_words = (n_img + 31) / 32;
  L.with_conf = with_conf; L.with_preselect = with_preselect;
  const size_t N = (size_t)n_images, NC = N * (size_t)n_img;
  size_t o = 0;
  auto block = [&o](size_t bytes) { const size_t at = o; o = b200_align_up(o + bytes, 256); return at; };
  L.counts = block(sizeof(int32_t) * N);
  if (with_preselect) { L.pre_count = block(sizeof(int) * N); L.pre_elig = block(sizeof(int) * N); }
  L.bitmap = block(sizeof(uint32_t) * N * L.bitmap_words);
  L.box = block(sizeof(float4) * NC);
  L.score = block(sizeof(float) * NC);
  L.cls = block(sizeof(int32_t) * NC);
  if (with_conf) L.conf = block(sizeof(float) * NC);
  L.aidx = block(sizeof(uint32_t) * NC);
  L.pos = block(sizeof(int32_t) * N * (size_t)max_out);
  if (with_preselect) {
    L.pre_khi = block(sizeof(unsigned long long) * N);
    L.pre_keys = block(sizeof(unsigned long long) * N * NMS_PRE_CAP);
    L.pre_pos = block(sizeof(uint32_t) * N * NMS_PRE_CAP);
  }
  L.total = o;
  return L;
}

// The store in workspace `ws` laid out by L.  The pre-selection buffers are always laid out when asked for, but bound
// only when an image can have more than NMS_PRE_MIN_N candidates: a bound pre_keys is what runs the pre-selection.
static inline CandStore cand_bind(const CandLayout& L, unsigned char* ws, bool sel_idx) {
  const bool pre = L.with_preselect && L.n_img > NMS_PRE_MIN_N;
  CandStore s;
  s.box = reinterpret_cast<float4*>(ws + L.box);
  s.score = reinterpret_cast<float*>(ws + L.score);
  s.cls = reinterpret_cast<int32_t*>(ws + L.cls);
  s.aidx = reinterpret_cast<uint32_t*>(ws + L.aidx);
  s.conf = L.with_conf ? reinterpret_cast<float*>(ws + L.conf) : nullptr;
  s.counts = reinterpret_cast<int32_t*>(ws + L.counts);
  s.bitmap = sel_idx ? reinterpret_cast<uint32_t*>(ws + L.bitmap) : nullptr;
  s.bitmap_words = L.bitmap_words; s.n_img = L.n_img;
  s.pos = reinterpret_cast<int32_t*>(ws + L.pos);
  s.pre_keys = pre ? reinterpret_cast<unsigned long long*>(ws + L.pre_keys) : nullptr;
  s.pre_pos = pre ? reinterpret_cast<uint32_t*>(ws + L.pre_pos) : nullptr;
  s.pre_count = pre ? reinterpret_cast<int*>(ws + L.pre_count) : nullptr;
  s.pre_elig = pre ? reinterpret_cast<int*>(ws + L.pre_elig) : nullptr;
  s.pre_khi = pre ? reinterpret_cast<unsigned long long*>(ws + L.pre_khi) : nullptr;
  return s;
}

// Appends the warp's lanes with `pass` set, grouped by image: one atomicAdd on counts[] per (warp, image), a lane's slot
// from its rank among the lanes of its image.  columns(slot) writes the caller's columns; the anchor index and the
// bitmap bit are written here.
template <class Columns>
__device__ __forceinline__ void warp_append_by_image(const CandStore& s, bool pass, int img, uint32_t aidx, Columns columns) {
  const int lane = threadIdx.x & 31;
  uint32_t todo = __ballot_sync(0xffffffffu, pass);
  while (todo) {
    const int leader = __ffs(todo) - 1;
    const int limg = __shfl_sync(0xffffffffu, img, leader);
    const uint32_t grp = __ballot_sync(0xffffffffu, pass && img == limg);
    int base = 0;
    if (lane == leader) base = atomicAdd(&s.counts[limg], __popc(grp));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (pass && img == limg) {
      const size_t slot = (size_t)limg * s.n_img + base + __popc(grp & ((1u << lane) - 1u));
      columns(slot);
      s.aidx[slot] = aidx;
      if (s.bitmap) atomicOr(&s.bitmap[(size_t)limg * s.bitmap_words + (aidx >> 5)], 1u << (aidx & 31u));
    }
    todo &= ~grp;
  }
}

// ---- NMS output tail of a finalize kernel (one CTA per image) ----
// The NMS segment of image img: its row of the store, with the classes for per-class NMS only.
__device__ __forceinline__ NmsSegment cand_segment(const CandStore& s, int img, bool with_classes) {
  const size_t base = (size_t)img * s.n_img;
  NmsSegment seg;
  seg.boxes = reinterpret_cast<const float*>(s.box + base);
  seg.scores = s.score + base;
  seg.classes = with_classes ? s.cls + base : nullptr;
  seg.order_id = s.aidx + base;
  seg.n = s.counts[img];
  return seg;
}

// After the NMS (wprefix reuses its shared memory): exclusive prefix popcount of image img's bitmap words, one pass by
// warp 0 (a few thousand words at most).  Does nothing without a bitmap.
__device__ __forceinline__ void cand_word_prefix(const CandStore& s, int img, uint32_t* wprefix) {
  if (!s.bitmap) return;
  const uint32_t* bm = s.bitmap + (size_t)img * s.bitmap_words;
  if (threadIdx.x < 32) {
    uint32_t run = 0;
    for (int w0 = 0; w0 < s.bitmap_words; w0 += 32) {
      const int w = w0 + (int)threadIdx.x;
      const int c = (w < s.bitmap_words) ? __popc(bm[w]) : 0;
      const int inc = warp_scan_incl(c);
      if (w < s.bitmap_words) wprefix[w] = run + (uint32_t)(inc - c);
      run += (uint32_t)__shfl_sync(0xffffffffu, inc, 31);
    }
  }
  __syncthreads();
}

// sel_idx of anchor index a of image img: its rank among the image's candidates, which is its position in the
// reference's compacted list
__device__ __forceinline__ int32_t cand_sel_idx(const CandStore& s, int img, const uint32_t* wprefix, uint32_t a) {
  const uint32_t wv = s.bitmap[(size_t)img * s.bitmap_words + (a >> 5)];
  return (int32_t)(wprefix[a >> 5] + __popc(wv & ((1u << (a & 31u)) - 1u)));
}

// dynamic shared memory of a finalize kernel: the NMS, then the word prefix in the same bytes
static inline size_t cand_finalize_smem_bytes(const CandStore& s, int max_out) {
  const size_t nms = nms_smem_bytes(max_out), prefix = (size_t)s.bitmap_words * 4;
  return nms < prefix ? prefix : nms;
}

// runs CALL(METRIC) with the runtime metric as a compile-time constant
#define NMS_DISPATCH_METRIC(metric, CALL)                               \
  switch (metric) {                                                     \
    case B200_METRIC_YOLO_IOU: { CALL(B200_METRIC_YOLO_IOU); } break;   \
    case B200_METRIC_YOLO_DIOU: { CALL(B200_METRIC_YOLO_DIOU); } break; \
    case B200_METRIC_YOLO_CIOU: { CALL(B200_METRIC_YOLO_CIOU); } break; \
    case B200_METRIC_EFF_IOU: { CALL(B200_METRIC_EFF_IOU); } break;     \
    case B200_METRIC_EFF_GIOU: { CALL(B200_METRIC_EFF_GIOU); } break;   \
    case B200_METRIC_EFF_DIOU: { CALL(B200_METRIC_EFF_DIOU); } break;   \
    default: { CALL(B200_METRIC_EFF_CIOU); } break;                     \
  }
