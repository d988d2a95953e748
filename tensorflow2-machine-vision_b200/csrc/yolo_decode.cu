// yolo_decode.cu — YOLOv3/v4 head decode + threshold filter + per-class NMS, fused post-processing.
//
// Replaces GetBoxes (utils/tf_yolo_utils.py:129-167) and GetNMSBoxes (:169-269) of the reference, with the
// B == 1 semantics of the reference applied per image (the reference flattens the batch, tyu:163-166).
//
// Kernel 1  yolo_decode_filter_kernel  (HBM-read bound: every head byte is read exactly once)
//   * each level tensor is treated as a flat array of records of RF = 5+C floats; a warp owns tiles of 32
//     records staged through its own WarpSlabRing (bulkcopy.cuh: one bulk copy per tile, a plain copy for a level's
//     ragged tail); 16 warps per SM, each with its own tile in flight;
//   * lane <-> record; the stride RF between lanes is odd for the 85-float COCO record so the column reads are
//     bank-conflict free; conf is thresholded first, then the class maximum is found on raw logits and the
//     sigmoid is evaluated only for logits inside a guard band of the maximum (max / first-argmax are taken
//     in sigmoid space, exactly as tf.reduce_max / tf.argmax of sigmoid(classes) do; detmath's sigmoid is not
//     monotone at ulp level, see oracle/DETMATH_REPORT.md);
//   * survivors (valid box, conf > thr, score > thr: strict, tyu:163,191-192) are appended per image to the candidate
//     store (CandStore, nms.cuh: its workspace layout, the warp-aggregated append and the NMS output tail live there,
//     shared with effdet.cu; YOLO adds the conf column).  Append order is arbitrary; each candidate carries its
//     flat anchor index (level-major, then h, w, a) which is monotone in the reference's compaction order, so it
//     serves as the NMS tie-break id and as the rank source for `sel_idx`.
// Kernel 2  yolo_nms_finalize_kernel  (one CTA per image): nms.cuh greedy NMS + gather of the five outputs,
//   recomputing sigmoid(classes) for the <= max_out selected rows straight from the head tensors.
#include <cmath>
#include "nms.cuh"
#include "bulkcopy.cuh"

#define YD_MAX_LEVELS 3
#define YD_STAGES 1

struct YoloLevels {
  const float* head[YD_MAX_LEVELS];
  int h[YD_MAX_LEVELS], w[YD_MAX_LEVELS];
  int rec_per_img[YD_MAX_LEVELS];   // h*w*A
  int anchor_base[YD_MAX_LEVELS];   // flat anchor index of the level's first record within an image
  long long total_rec[YD_MAX_LEVELS];  // B*h*w*A
  long long tile_base[YD_MAX_LEVELS + 1];  // first global tile index of each level
  float anc_w[YD_MAX_LEVELS][8], anc_h[YD_MAX_LEVELS][8];  // anchors_wh / image_wh (fp32 division, tyu:185)
  // lowest tw / th for which the decoded box is certainly valid (w >= 4e-7 so that x + w/2 > x - w/2 in fp32 for any
  // centre in [0,1]); together with t <= 80 (no overflow) and non-NaN tx, ty the filter can skip the decode
  float tmin_w[YD_MAX_LEVELS][8], tmin_h[YD_MAX_LEVELS][8];
};

struct YoloDecodeParams {
  YoloLevels lv;
  int B, A, C, RF;
  float conf_thr, score_thr;
  float conf_lo, conf_hi;  // logits below / above which sigmoid(conf) > conf_thr is decided without the sigmoid
  uint32_t magic_a;        // floor(2^32/A)+1 (0 for A == 1): rin / A == umulhi(rin, magic_a) for rin * A < 2^32
  CandStore st;            // box is left to the NMS pass (decode on demand)
};

// max and first-argmax of sigmoid(x_c), c in [0,C), for the warp's 32 records (lane <-> record, stride RF in shared
// memory, conflict-free).  One pass per lane keeps the largest logit with its first index and the second largest
// value (four independent chains).  When the runner-up is outside the guard band of the maximum its sigmoid is
// certainly smaller and the answer is (sigmoid(m1), i1): for -80 < m < 8, d ln(sigmoid)/dx >= 3.3e-4, so logits
// below m - 0.01 are > 3.3e-6 relative below sigmoid(m) while detmath's sigmoid is within 2.4 ulp = 2.9e-7 of exact
// (oracle/DETMATH_REPORT.md; it is not monotone at ulp level, which is why the band exists).  Otherwise (a few per
// cent of the records) the whole warp evaluates that record's in-band logits and takes max / first-argmax in sigmoid
// space, exactly as tf.reduce_max / tf.argmax of sigmoid(classes) do.
__device__ __forceinline__ void class_max_sigmoid_warp(const float* __restrict__ slab, int RF, int C, bool want, int lane,
                                                       float& best_s, int& best_c) {
  const float* __restrict__ cls = slab + lane * RF + 5;
  bool slow = false;
  float lo = -INFINITY;
  if (want) {
    float a[4], m2[4], nan_acc = 0.0f;
    int ix[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { a[k] = -INFINITY; m2[k] = -INFINITY; ix[k] = C; }
    int c = 0;
    for (; c + 4 <= C; c += 4) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float x = cls[c + k];
        nan_acc = __fmaf_rn(x, 0.0f, nan_acc);            // NaN once any logit is NaN or +-inf
        m2[k] = fmaxf(m2[k], fminf(a[k], x));
        const bool g = x > a[k];                            // strict: the first index of a chain's maximum stays
        a[k] = g ? x : a[k];
        ix[k] = g ? c + k : ix[k];
      }
    }
    for (; c < C; ++c) {
      const float x = cls[c];
      nan_acc = __fmaf_rn(x, 0.0f, nan_acc);
      m2[0] = fmaxf(m2[0], fminf(a[0], x));
      const bool g = x > a[0];
      a[0] = g ? x : a[0];
      ix[0] = g ? c : ix[0];
    }
    // merge the chains: largest value, lowest index on ties; runner-up = largest of the chains' runner-ups and of
    // the chain maxima that lost
    float m1 = a[0], r2 = m2[0];
    int i1 = ix[0];
#pragma unroll
    for (int k = 1; k < 4; ++k) {
      const bool g = (a[k] > m1) || (a[k] == m1 && ix[k] < i1);
      r2 = fmaxf(r2, fmaxf(m2[k], g ? m1 : a[k]));
      m1 = g ? a[k] : m1;
      i1 = g ? ix[k] : i1;
    }
    const bool banded = (m1 < 8.0f) && (m1 > -80.0f);
    lo = banded ? (m1 - 0.01f) : -INFINITY;
    slow = !(nan_acc == 0.0f) || !(r2 < lo) || i1 >= C;
    best_s = m1;  // sigmoid applied below
    best_c = i1;
  }
  if (want && !slow) best_s = dm_sigmoidf(best_s);
  // cooperative exact path, one record at a time
  uint32_t todo = __ballot_sync(0xffffffffu, want && slow);
  while (todo) {
    const int src = __ffs(todo) - 1;
    todo &= todo - 1u;
    const float lo_s = __shfl_sync(0xffffffffu, lo, src);
    const float* __restrict__ rc = slab + src * RF + 5;
    // serial semantics being reproduced: walk c upwards over the in-band logits (x >= lo or NaN); the first one
    // initialises (s, c) even when its sigmoid is NaN; later ones replace it only when s > best
    float ls = 0.0f;
    int lc = 0x7fffffff, lfirst = 0x7fffffff;
    bool lfirst_nan = false;
    for (int c = lane; c < C; c += 32) {
      const float x = rc[c];
      if (x >= lo_s || x != x) {
        const float sg = dm_sigmoidf(x);
        if (lfirst == 0x7fffffff) { lfirst = c; lfirst_nan = sg != sg; }
        if (sg == sg && (lc == 0x7fffffff || sg > ls)) { ls = sg; lc = c; }
      }
    }
    int first = lfirst;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
    const bool first_is_nan = __any_sync(0xffffffffu, lfirst == first && first != 0x7fffffff && lfirst_nan);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float os = __shfl_xor_sync(0xffffffffu, ls, o);
      const int oc = __shfl_xor_sync(0xffffffffu, lc, o);
      const bool take = (oc != 0x7fffffff) && (lc == 0x7fffffff || os > ls || (os == ls && oc < lc));
      ls = take ? os : ls;
      lc = take ? oc : lc;
    }
    if (lane == src) {
      if (first == 0x7fffffff) { best_s = 0.0f; best_c = 0; }               // no in-band logit at all (cannot happen for C >= 1)
      else if (first_is_nan || lc == 0x7fffffff) { best_s = __int_as_float(0x7fc00000); best_c = first; }
      else { best_s = ls; best_c = lc; }
    }
  }
}

struct Decoded { float x1, y1, x2, y2; bool valid; };

__device__ __forceinline__ Decoded decode_box(float tx, float ty, float tw, float th, int gx, int gy, int W, int H,
                                              float aw, float ah) {
  // tyu:153-161: xy = (sigmoid(t)+grid)/grid_wh; wh = exp(t)*anchor (anchor already /image_wh); inf -> 0
  Decoded d;
  float x = DM_DIV(DM_ADD(dm_sigmoidf(tx), (float)gx), (float)W);
  float y = DM_DIV(DM_ADD(dm_sigmoidf(ty), (float)gy), (float)H);
  float w = DM_MUL(dm_expf(tw), aw);
  float h = DM_MUL(dm_expf(th), ah);
  if (dm_isinf(w)) w = 0.0f;
  if (dm_isinf(h)) h = 0.0f;
  float hw = DM_DIV(w, 2.0f), hh = DM_DIV(h, 2.0f);
  d.x1 = DM_SUB(x, hw); d.y1 = DM_SUB(y, hh); d.x2 = DM_ADD(x, hw); d.y2 = DM_ADD(y, hh);
  d.valid = (d.x2 > d.x1) && (d.y2 > d.y1);
  return d;
}

template <bool EARLY>   // EARLY: a warp refills its slab before its append (atomic + stores) instead of after it
__global__ void __launch_bounds__(512, 1) yolo_decode_filter_kernel(YoloDecodeParams p) {
  extern __shared__ __align__(128) unsigned char yd_smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int warps_per_cta = blockDim.x >> 5;
  const int RF = p.RF;
  WarpSlabRing<YD_STAGES> ring(yd_smem, RF);

  const long long n_tiles = p.lv.tile_base[YD_MAX_LEVELS];
  const long long gwarp = (long long)blockIdx.x * warps_per_cta + warp;
  const long long gstride = (long long)gridDim.x * warps_per_cta;

  // issue the load of `tile` into stage s
  auto issue = [&](long long tile, int s) {
    int l = 0;
#pragma unroll
    for (int k = 1; k < YD_MAX_LEVELS; ++k) if (tile >= p.lv.tile_base[k]) l = k;
    const long long rec0 = (tile - p.lv.tile_base[l]) * 32;
    const long long remain = p.lv.total_rec[l] - rec0;
    ring.issue(s, p.lv.head[l] + rec0 * RF, remain < 32 ? (int)remain : 32, RF);
  };

  long long t_issue = gwarp;
#pragma unroll
  for (int s = 0; s < YD_STAGES; ++s) {
    if (t_issue < n_tiles) issue(t_issue, s);
    t_issue += gstride;
  }
  for (long long tile = gwarp; tile < n_tiles; tile += gstride) {
    ring.wait();
    const float* slab = ring.slab(ring.stage);
    int l = 0;
#pragma unroll
    for (int k = 1; k < YD_MAX_LEVELS; ++k) if (tile >= p.lv.tile_base[k]) l = k;
    const long long rec = (tile - p.lv.tile_base[l]) * 32 + lane;
    const bool in_range = rec < p.lv.total_rec[l];
    const float* r = slab + lane * RF;
    bool pass = false;
    int img = 0;
    float score = 0.f, conf = 0.f;
    int cls = 0;
    uint32_t aidx = 0;
    bool want = false;
    if (in_range) {
      // sigmoid(conf) > conf_thr (tyu:191), decided in logit space outside a narrow band around logit(conf_thr)
      conf = r[4];
      if (conf > p.conf_hi) want = true;
      else if (conf >= p.conf_lo) want = dm_sigmoidf(conf) > p.conf_thr;  // NaN fails both comparisons: not wanted
    }
    class_max_sigmoid_warp(slab, RF, p.C, want, lane, score, cls);
    if (want && score > p.score_thr) {
      const int rpi = p.lv.rec_per_img[l];
      // 32-bit division when the level has fewer than 2^31 records (always, short of ~100k-image batches)
      img = (p.lv.total_rec[l] < 0x7fffffffLL) ? (int)((uint32_t)rec / (uint32_t)rpi) : (int)(rec / rpi);
      const int rin = (int)(rec - (long long)img * rpi);
      const int cell = p.magic_a ? (int)__umulhi((uint32_t)rin, p.magic_a) : rin, a = rin - cell * p.A;  // rin / A
      // the box itself is decoded by the NMS pass, and only for the candidates it looks at; here only its validity
      // (x2 > x1 and y2 > y1, tyu:163) is needed: certain inside the safe logit range, exact decode otherwise
      const float tx = r[0], ty = r[1], tw = r[2], th = r[3];
      bool valid = (tw >= p.lv.tmin_w[l][a]) && (tw <= 80.0f) && (th >= p.lv.tmin_h[l][a]) && (th <= 80.0f) && (tx == tx) && (ty == ty);
      if (!valid) {
        const int W = p.lv.w[l], H = p.lv.h[l];
        const int gy = cell / W, gx = cell - gy * W;
        valid = decode_box(tx, ty, tw, th, gx, gy, W, H, p.lv.anc_w[l][a], p.lv.anc_h[l][a]).valid;
      }
      if (valid) {
        pass = true;
        aidx = (uint32_t)(p.lv.anchor_base[l] + rin);
      }
    }
    // Every lane is done reading the slab: refill it NOW, so that the copy of the next tile is in flight during the append
    // below (an atomic round trip to L2 plus the stores — 9 % of the warp's cycle when the copy was issued after it).
    if (EARLY) {
      __syncwarp();
      if (t_issue < n_tiles) issue(t_issue, ring.stage);
      t_issue += gstride;
    }
    warp_append_by_image(p.st, pass, img, aidx, [&](size_t slot) {
      p.st.score[slot] = score;
      p.st.cls[slot] = cls;
      p.st.conf[slot] = conf;  // the logit; the sigmoid is applied to the emitted rows only
    });
    if (!EARLY) {
      __syncwarp();  // every lane is done reading the slab before it is refilled
      if (t_issue < n_tiles) issue(t_issue, ring.stage);
      t_issue += gstride;
    }
    ring.advance();
  }
}

struct YoloFinalizeParams {
  YoloLevels lv;
  int B, A, C, RF;
  NmsConfig cfg;
  CandStore st;      // box is written by the NMS pass (decode on demand)
  // outputs, all [B, max_out, ...]
  float* out_boxes; int32_t* out_cls; float* out_score; float* out_classes; float* out_conf;
  int32_t* out_sel_idx; int32_t* out_sel_anchor; int32_t* out_count;
};

// Decode-on-demand for NMS: candidate `pos` of the image -> its record in the head tensor -> decode_box; the result is
// written back to the candidate store so that the emitted rows can be copied out afterwards.
struct YoloLazyBox {
  static constexpr bool kKeyCache = true;   // a 416x416 image has ~5 k candidates: its selection passes run from registers
  static constexpr int kMode = B200_NMS_BY_CLASS;
  static constexpr bool kSampleRange = false;
  const YoloLevels* lv;
  int img, A, RF;
  float4* cand_box;  // this image's slice
  __device__ __forceinline__ float4 operator()(const NmsSegment& seg, uint32_t pos) const {
    const int a_flat = (int)seg.order_id[pos];
    int l = 0;
#pragma unroll
    for (int j = 1; j < YD_MAX_LEVELS; ++j) if (a_flat >= lv->anchor_base[j]) l = j;
    const int rin = a_flat - lv->anchor_base[l];
    const float* r = lv->head[l] + ((long long)img * lv->rec_per_img[l] + rin) * RF;
    const int cell = rin / A, a = rin - cell * A;
    const int W = lv->w[l], H = lv->h[l];
    const int gy = cell / W, gx = cell - gy * W;
    const Decoded d = decode_box(__ldg(r), __ldg(r + 1), __ldg(r + 2), __ldg(r + 3), gx, gy, W, H, lv->anc_w[l][a], lv->anc_h[l][a]);
    const float4 b = make_float4(d.x1, d.y1, d.x2, d.y2);
    cand_box[pos] = b;
    return b;
  }
};

template <int METRIC, int THREADS>
__global__ void __launch_bounds__(THREADS, NMS_THREADS / THREADS) yolo_nms_finalize_kernel(YoloFinalizeParams p) {
  extern __shared__ __align__(16) unsigned char nms_smem[];
  const int img = blockIdx.x;
  const size_t cbase = (size_t)img * p.st.n_img;
  int32_t* pos = p.st.pos + (size_t)img * p.cfg.max_out;
  YoloLazyBox lazy;
  lazy.lv = &p.lv; lazy.img = img; lazy.A = p.A; lazy.RF = p.RF; lazy.cand_box = p.st.box + cbase;
  const int kept = nms_run_segment<METRIC, YoloLazyBox, THREADS>(cand_segment(p.st, img, true), p.cfg, pos, nms_smem, nullptr, lazy);
  __syncthreads();
  if (threadIdx.x == 0) p.out_count[img] = kept;
  const size_t obase = (size_t)img * p.cfg.max_out;
  uint32_t* wprefix = reinterpret_cast<uint32_t*>(nms_smem);
  cand_word_prefix(p.st, img, wprefix);
  for (int k = threadIdx.x; k < kept; k += blockDim.x) {
    const int q = pos[k];
    reinterpret_cast<float4*>(p.out_boxes)[obase + k] = p.st.box[cbase + q];
    p.out_cls[obase + k] = p.st.cls[cbase + q];
    p.out_score[obase + k] = p.st.score[cbase + q];
    p.out_conf[obase + k] = dm_sigmoidf(p.st.conf[cbase + q]);
    const uint32_t a = p.st.aidx[cbase + q];
    pos[k] = (int32_t)a;   // from here on the scratch row holds flat anchor indices: yolo_classes_kernel needs no candidate lookup
    if (p.out_sel_anchor) p.out_sel_anchor[obase + k] = (int32_t)a;
    if (p.out_sel_idx) p.out_sel_idx[obase + k] = cand_sel_idx(p.st, img, wprefix, a);
  }
}

// sigmoid(classes) rows of the selected boxes, read back from the head tensors (tyu:140,265).  A separate launch
// so the B*max_out*C sigmoids spread over the whole GPU instead of serialising inside the per-image NMS CTAs.
// LPR lanes per row: the kernel is bound by the issue of the deterministic sigmoid (~60 instructions), so the lanes that
// idle in a row's last round are the cost — 80 classes on 32 lanes waste one round in six, on 16 lanes (two rows per
// warp) none.
template <int LPR>
__global__ void __launch_bounds__(256) yolo_classes_kernel(YoloFinalizeParams p) {
  constexpr int RPW = 32 / LPR, NJ = 128 / LPR;
  const int sub = threadIdx.x & (LPR - 1);
  const int row = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * RPW + ((threadIdx.x & 31) / LPR);  // row = img * max_out + k
  if (row >= p.B * p.cfg.max_out) return;
  const int img = row / p.cfg.max_out, k = row - img * p.cfg.max_out;
  // flat anchor index, left by the NMS kernel; fetched together with the count (rows past the count hold stale values)
  const uint32_t a = (uint32_t)__ldcg(p.st.pos + (size_t)img * p.cfg.max_out + k);
  if (k >= __ldcg(p.out_count + img)) return;
  int l = 0;
#pragma unroll
  for (int j = 1; j < YD_MAX_LEVELS; ++j) if ((int)a >= p.lv.anchor_base[j]) l = j;
  const long long rec = (long long)img * p.lv.rec_per_img[l] + ((int)a - p.lv.anchor_base[l]);
  const float* src = p.lv.head[l] + rec * p.RF + 5;
  float* dst = p.out_classes + (size_t)row * p.C;
  // the (cold) logits of up to 128 classes are fetched before the first sigmoid starts
  float x[NJ];
#pragma unroll
  for (int j = 0; j < NJ; ++j) x[j] = (sub + LPR * j < p.C) ? __ldg(src + sub + LPR * j) : 0.0f;
#pragma unroll
  for (int j = 0; j < NJ; ++j) if (sub + LPR * j < p.C) dst[sub + LPR * j] = dm_sigmoidf(x[j]);
  for (int c = sub + 128; c < p.C; c += LPR) dst[c] = dm_sigmoidf(__ldg(src + c));
}

// ---- dense decode for the stand-alone GetBoxes shim ---------------------------------------------
// One warp per record: boxes/conf/sigmoid(classes)/valid for every anchor of one level, no filtering.
__global__ void yolo_decode_dense_kernel(const float* __restrict__ head, long long total_rec, int H, int W, int A,
                                         int C,
                                         const float* __restrict__ anc_wh, float* __restrict__ boxes,
                                         float* __restrict__ conf, float* __restrict__ classes,
                                         unsigned char* __restrict__ valid) {
  const int RF = 5 + C;
  const int lane = threadIdx.x & 31;
  long long rec = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const long long stride = (long long)gridDim.x * (blockDim.x >> 5);
  const int rpi = H * W * A;
  for (; rec < total_rec; rec += stride) {
    const float* r = head + rec * RF;
    for (int c = lane; c < C; c += 32) classes[rec * C + c] = dm_sigmoidf(__ldg(r + 5 + c));
    if (lane == 0) {
      const int rin = (int)(rec % rpi);
      const int cell = rin / A, a = rin - cell * A;
      const int gy = cell / W, gx = cell - gy * W;
      Decoded d = decode_box(__ldg(r), __ldg(r + 1), __ldg(r + 2), __ldg(r + 3), gx, gy, W, H, anc_wh[2 * a], anc_wh[2 * a + 1]);
      boxes[rec * 4 + 0] = d.x1; boxes[rec * 4 + 1] = d.y1; boxes[rec * 4 + 2] = d.x2; boxes[rec * 4 + 3] = d.y2;
      conf[rec] = dm_sigmoidf(__ldg(r + 4));
      valid[rec] = d.valid ? 1 : 0;
    }
  }
}

// ---- host side ---------------------------------------------------------------------------------
static int fill_levels(YoloLevels& lv, const float* const heads[3], const int32_t hw[6], int B, int A, int C,
                       const float* anchors_wh_host, const float* image_wh_host) {
  long long tb = 0;
  int ab = 0;
  for (int l = 0; l < YD_MAX_LEVELS; ++l) {
    lv.head[l] = heads[l];
    lv.h[l] = hw[2 * l];
    lv.w[l] = hw[2 * l + 1];
    lv.rec_per_img[l] = lv.h[l] * lv.w[l] * A;
    lv.anchor_base[l] = ab;
    ab += lv.rec_per_img[l];
    lv.total_rec[l] = (long long)B * lv.rec_per_img[l];
    lv.tile_base[l] = tb;
    tb += (lv.total_rec[l] + 31) / 32;
    for (int a = 0; a < A; ++a) {
      lv.anc_w[l][a] = anchors_wh_host[(l * A + a) * 2 + 0] / image_wh_host[0];
      lv.anc_h[l][a] = anchors_wh_host[(l * A + a) * 2 + 1] / image_wh_host[1];
      // w = exp(tw) * anchor >= 4e-7 (twice the 2e-7 that guarantees x + w/2 > x - w/2 for x in [0,1]); anchors that
      // are not positive and finite never qualify
      const double aw = lv.anc_w[l][a], ah = lv.anc_h[l][a];
      lv.tmin_w[l][a] = (aw > 0.0 && aw < 1e30) ? (float)(log(4e-7 / aw) + 1e-3) : INFINITY;
      lv.tmin_h[l][a] = (ah > 0.0 && ah < 1e30) ? (float)(log(4e-7 / ah) + 1e-3) : INFINITY;
    }
  }
  lv.tile_base[YD_MAX_LEVELS] = tb;
  return ab;
}

extern "C" size_t b200_yolo_decode_nms_workspace_bytes(const int32_t hw[6], int B, int A, int max_out) {
  int n_img = 0;
  for (int l = 0; l < 3; ++l) n_img += hw[2 * l] * hw[2 * l + 1] * A;
  return cand_layout(B, n_img, max_out, true, false).total;
}

extern "C" int b200_yolo_decode_nms(const float* const heads[3], const int32_t hw[6], int B, int A, int C,
                                    const float* anchors_wh_host, const float* image_wh_host, float conf_thr,
                                    float score_thr, float iou_thr, int metric, int max_out, float* out_boxes,
                                    int32_t* out_class_id, float* out_score, float* out_classes, float* out_conf,
                                    int32_t* out_sel_idx, int32_t* out_sel_anchor, int32_t* out_count,
                                    void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  B200_REQUIRE(heads && hw && anchors_wh_host && image_wh_host, B200_ERR_BAD_ARG, "b200_yolo_decode_nms: null argument");
  B200_REQUIRE(B >= 0 && A >= 1 && A <= 8 && C >= 1 && C <= 1019, B200_ERR_BAD_ARG,
               "b200_yolo_decode_nms: unsupported shape B=%d A=%d C=%d", B, A, C);
  B200_REQUIRE(metric >= B200_METRIC_YOLO_IOU && metric <= B200_METRIC_YOLO_CIOU, B200_ERR_BAD_ARG,
               "b200_yolo_decode_nms: iou_type must be iou/diou/ciou (metric %d)", metric);
  B200_REQUIRE(max_out >= 1 && max_out <= NMS_MAX_OUT_LIMIT, B200_ERR_UNSUPPORTED, "b200_yolo_decode_nms: max_out %d outside [1,%d]", max_out, NMS_MAX_OUT_LIMIT);
  if (B == 0) return B200_OK;
  B200_REQUIRE(out_boxes && out_class_id && out_score && out_conf && out_count, B200_ERR_BAD_ARG, "b200_yolo_decode_nms: null output");
  for (int l = 0; l < 3; ++l) {
    B200_REQUIRE(heads[l] != nullptr && hw[2 * l] > 0 && hw[2 * l + 1] > 0, B200_ERR_BAD_ARG, "b200_yolo_decode_nms: bad level %d", l);
    B200_REQUIRE((reinterpret_cast<uintptr_t>(heads[l]) & 15) == 0, B200_ERR_BAD_ARG, "b200_yolo_decode_nms: head %d not 16-byte aligned", l);
  }
  B200_REQUIRE((reinterpret_cast<uintptr_t>(out_boxes) & 15) == 0, B200_ERR_BAD_ARG, "b200_yolo_decode_nms: out_boxes not 16-byte aligned");
  YoloDecodeParams dp;
  const int n_img = fill_levels(dp.lv, heads, hw, B, A, C, anchors_wh_host, image_wh_host);
  const CandLayout ws = cand_layout(B, n_img, max_out, true, false);
  B200_REQUIRE(workspace && workspace_bytes >= ws.total, B200_ERR_WORKSPACE,
               "b200_yolo_decode_nms: workspace %zu < required %zu", workspace_bytes, ws.total);
  B200_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, B200_ERR_BAD_ARG, "b200_yolo_decode_nms: workspace not 256-byte aligned");
  unsigned char* wsb = static_cast<unsigned char*>(workspace);
  dp.B = B; dp.A = A; dp.C = C; dp.RF = 5 + C;
  dp.conf_thr = conf_thr; dp.score_thr = score_thr;
  dp.magic_a = A == 1 ? 0u : (uint32_t)((1ull << 32) / (unsigned long long)A + 1ull);
  // sigmoid(x) > conf_thr is certain for x > logit(thr) + d and certainly false for x < logit(thr) - d, with d ten times
  // the 2.4-ulp error of the deterministic sigmoid divided by the slope thr(1-thr); thresholds near 0 or 1 (or outside
  // (0,1)) always take the exact comparison
  dp.conf_lo = -INFINITY; dp.conf_hi = INFINITY;
  if (conf_thr >= 1e-3f && conf_thr <= 1.0f - 1e-3f) {
    const double t = log((double)conf_thr / (1.0 - (double)conf_thr));
    const double d = 3e-6 / ((double)conf_thr * (1.0 - (double)conf_thr)) + 1e-6 * fabs(t);
    dp.conf_lo = (float)(t - d); dp.conf_hi = (float)(t + d);
  }
  dp.st = cand_bind(ws, wsb, out_sel_idx != nullptr);
  B200_CUDA(cudaMemsetAsync(wsb, 0, ws.zeroed(out_sel_idx != nullptr), stream));

  using Ring = WarpSlabRing<YD_STAGES>;
  int warps = 16;  // one tile in flight per warp; the warps of an SM overlap each other's loads
  while (warps > 1 && Ring::smem_bytes(warps, dp.RF) > 200 * 1024) warps >>= 1;
  // a single image has fewer tiles than the GPU has warp slots: spread them (one warp per scheduler finishes its tile sooner)
  while (warps > 2 && dp.lv.tile_base[YD_MAX_LEVELS] <= (long long)(warps / 2) * b200_sm_count()) warps >>= 1;
  const size_t smem1 = Ring::smem_bytes(warps, dp.RF);
  B200_REQUIRE(smem1 <= 220 * 1024, B200_ERR_UNSUPPORTED, "b200_yolo_decode_nms: record too large (C=%d)", C);

  const long long n_tiles = dp.lv.tile_base[YD_MAX_LEVELS];
  const int grid = Ring::grid(n_tiles, warps, b200_sm_count());
  // Refilling a warp's slab before its append keeps one more copy in flight: -3 % for the call on its own at any size, and
  // for the fused evaluation step at 512 images; at 64 images per GPU the same step is 3 % SLOWER with it (the filter then
  // takes DRAM bandwidth from the loss chain that shares the GPU, and that chain is the longer one there).  Long streams
  // (>= 32 tiles per warp) refill early, short ones late.
  if (n_tiles >= 32ll * grid * warps) {
    B200_CUDA(cudaFuncSetAttribute(yolo_decode_filter_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
    yolo_decode_filter_kernel<true><<<grid, warps * 32, smem1, stream>>>(dp);
  } else {
    B200_CUDA(cudaFuncSetAttribute(yolo_decode_filter_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
    yolo_decode_filter_kernel<false><<<grid, warps * 32, smem1, stream>>>(dp);
  }
  B200_LAUNCH_CHECK();

  YoloFinalizeParams fp;
  fp.lv = dp.lv; fp.B = B; fp.A = A; fp.C = C; fp.RF = dp.RF; fp.st = dp.st;
  fp.cfg.metric = metric; fp.cfg.mode = B200_NMS_BY_CLASS; fp.cfg.iou_thr = iou_thr; fp.cfg.score_thr = 0.f;
  fp.cfg.use_score_thr = 0; fp.cfg.max_out = max_out;
  fp.out_boxes = out_boxes; fp.out_cls = out_class_id; fp.out_score = out_score; fp.out_classes = out_classes;
  fp.out_conf = out_conf; fp.out_sel_idx = out_sel_idx; fp.out_sel_anchor = out_sel_anchor; fp.out_count = out_count;
  // one 1024-thread CTA per SM gives the lowest latency; batches that need more than one wave use 512-thread CTAs,
  // two per SM (the shared-memory footprint allows it up to max_out ~ 500)
  const size_t smem2 = cand_finalize_smem_bytes(fp.st, max_out);
  const bool half_ctas = (B > b200_sm_count()) && (2 * (smem2 + 1024) <= 227 * 1024);
#define YD_LAUNCH(M)                                                                                                   \
  if (half_ctas) {                                                                                                          \
    B200_CUDA(cudaFuncSetAttribute(yolo_nms_finalize_kernel<M, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2)); \
    yolo_nms_finalize_kernel<M, 512><<<B, 512, smem2, stream>>>(fp);                                                         \
  } else {                                                                                                                  \
    B200_CUDA(cudaFuncSetAttribute(yolo_nms_finalize_kernel<M, NMS_THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2)); \
    yolo_nms_finalize_kernel<M, NMS_THREADS><<<B, NMS_THREADS, smem2, stream>>>(fp);                                         \
  }
  NMS_DISPATCH_METRIC(metric, YD_LAUNCH)
#undef YD_LAUNCH
  B200_LAUNCH_CHECK();
  if (out_classes) {
    const long long rows = (long long)B * max_out;
    // half a warp per row when that leaves fewer idle lanes in the last round (80 classes: 5 x 16 against 3 x 32)
    // (a few hundred rows are latency-bound: a full warp per row has the shorter chain)
    if (rows >= 16384 && ((C + 15) / 16) * 16 < ((C + 31) / 32) * 32) yolo_classes_kernel<16><<<(int)((rows + 15) / 16), 256, 0, stream>>>(fp);
    else yolo_classes_kernel<32><<<(int)((rows + 7) / 8), 256, 0, stream>>>(fp);
    B200_LAUNCH_CHECK();
  }
  return B200_OK;
}

extern "C" int b200_yolo_decode_dense(const float* head, int B, int H, int W, int A, int C,
                                      const float* anchors_wh_norm_dev, float* boxes, float* conf, float* classes,
                                      unsigned char* valid, void* stream) {
  B200_REQUIRE(B >= 0 && H > 0 && W > 0 && A >= 1 && C >= 1, B200_ERR_BAD_ARG, "b200_yolo_decode_dense: bad shape");
  if (B == 0) return B200_OK;
  B200_REQUIRE(head && anchors_wh_norm_dev && boxes && conf && classes && valid, B200_ERR_BAD_ARG, "b200_yolo_decode_dense: null pointer");
  const long long total = (long long)B * H * W * A;
  long long blocks = (total + 7) / 8;
  long long cap = (long long)b200_sm_count() * 64;
  if (blocks > cap) blocks = cap;
  yolo_decode_dense_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(head, total, H, W, A, C, anchors_wh_norm_dev, boxes, conf,
                                                                         classes, valid);
  B200_LAUNCH_CHECK();
  return B200_OK;
}
