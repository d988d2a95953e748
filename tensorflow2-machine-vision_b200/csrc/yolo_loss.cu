// yolo_loss.cu — fused YOLOv3/v4 loss: GetLoss (utils/tf_yolo_utils.py:6-127) and its keras-yolo3 twin
// Yolov4Loss.call (losses/yolo_loss.py:85-159).
//
// The reference materialises ~20 (H,W,A,n_gt) broadcast temporaries per image inside a tf.while_loop; here
// the loss is three to four launches over the dense NHWC tensors, touching only the sectors the arithmetic needs:
//
//  K4a yolo_loss_scan_kernel     one CTA per 1024 consecutive anchor records of one (level, image): reads the obj
//      channel of y_true (one 32-byte sector per 340-byte record), stores it to a compact per-anchor array and appends
//      the records with obj != 0 (the ground-truth list, tyu:82) to the (image, level) object list.
//  K4a' yolo_loss_gtprep_kernel   a thread per object: the prepared GT box (corners, area, atan(w/h), log area) of the
//      ignore mask.
//  K4b yolo_loss_ignore_kernel    one CTA per 128 records: reads the 5 box/conf logits of every y_pred record, runs
//      the decode-free and approximate-IoU rejects against the GT list, queues the surviving (record, GT) pairs for
//      the exact decode (tyu:57-75) and exact metric (iou / diou / ciou, tiu:5-65), and accumulates
//      object_loss = obj*bce + (1-obj)*bce*ignore (tyu:111-114).  The trailing CTAs of its grid instead take a warp per
//      object and produce the xy, wh and class terms (tyu:107-118) from the full y_true / y_pred records.
//      This single-kernel form runs when y_pred is in pinned host memory (read in place over PCIe), when a level of
//      y_pred is not 16-byte aligned, or when a record holds fewer than 8 floats (C < 3).
//      Every other call (device-resident y_pred, every level 16-byte aligned, records of >= 8 floats) SPLITS the pass.
//      K4b-lean (yolo_loss_ignore_lean_kernel, 48 registers, 10 CTAs per SM) streams, applies the same rejects and only
//      QUEUES the records that some GT might still hit (~1 % of them); K4b-exact resolves the queue (a warp per record) at
//      the head of the widened K4c launch, its object-loss terms in 2^-32 fixed point so that the sum does not depend on
//      the order.  The launches of a dense call are then K4a (whose last CTA per (image, level) also does K4a'),
//      K4b-lean, K4c.
//  K4c yolo_loss_finalize_kernel  fixed-order fp64 reduction of the per-CTA partials -> parts[3][4] / batch,
//      loss = sum_l ((xy+wh)+obj)+cls in fp32 in the reference's order (tyu:120-125).  Deterministic run to run (the object lists are
//      put into ascending record order by K4a' before anything is summed over them).
//
// ignore = float(best < thr) with best = max_g metric(pred, gt_g) is evaluated as "no g with metric >= thr or
// metric NaN": tf.reduce_max propagates NaN and NaN < thr is False, so a NaN pair clears the ignore bit.
#include "yolo_targets.cuh"
#include "exchange.cuh"

#define YL_LEVELS 3
#define YL_CHUNK 256
#define YL_ICHUNK 128  // records (threads) per CTA of the ignore kernels

enum { YL_VARIANT_TF_YOLO_UTILS = 0, YL_VARIANT_KERAS_YOLO3 = 1 };

struct YlLevels {
  const float* y_true[YL_LEVELS];
  const float* y_pred[YL_LEVELS];
  int h[YL_LEVELS], w[YL_LEVELS], rec_per_img[YL_LEVELS], anchor_base[YL_LEVELS];
  int chunks_per_img[YL_LEVELS];
  int cta_base[YL_LEVELS + 1];
  int obj_chunks_per_img[YL_LEVELS];   // scan kernel: 4 records per thread
  int obj_cta_base[YL_LEVELS + 1];
  uint32_t magic_w[YL_LEVELS];         // floor(2^32/W)+1
  float anc_w[YL_LEVELS][8], anc_h[YL_LEVELS][8];  // pixels
};

struct YlParams {
  YlLevels lv;
  int B, A, C, RF, n_img;
  float img_w, img_h;  // divisors of the width / height channels (the variant decides the order, see yolo_loss_impl)
  float thr;
  int metric, variant;
  float* obj_compact;   // [B, n_img]
  float4* gt_box;       // [B, n_img] GT corners (level slices at anchor_base)
  float4* gt_aux;       // [B, n_img] area, atan(w/h), log(area), regular flag (1/0)
  float log_thr;        // log(thr)
  float logk[YL_LEVELS][8];  // log(anchor_w*anchor_h/(img_w*img_h)) per level/anchor
  float tmin_w[YL_LEVELS][8], tmin_h[YL_LEVELS][8];  // lowest tw/th for which the decode-free area bound holds
  uint32_t magic_a;           // floor(2^32/A)+1: n/A == umulhi(n, magic) for n*A < 2^32
  float* conf_grad;           // optional [level-major: B*anchor_base[l] + image*rec_per_img + rin]: d loss / d conf logit
  int32_t* obj_index;         // [B, n_img]: record index of each object-list / GT-list slot
  float inv_div;              // 1 / batch_divisor
  unsigned char* out_ignore;  // optional [B, n_img]: the ignore mask (1 = ignored/background), for parity tests
  // sparse-target mode (b200_yolo_loss_from_boxes: no dense y_true): per object slot the record's (x, y, w, h) and
  // class, and one obj bit per record
  const float4* sp_t;         // [B, n_img]
  const int32_t* sp_cls;      // [B, n_img]
  const uint32_t* obj_bits;   // [B, bits_words]
  int bits_words;
  int32_t* gt_count;    // [B, 3]
  unsigned int* scan_ticket;  // [B, 3] scan CTAs done per (image, level): the last one prepares that GT list (null: K4a' runs as a launch)
  // split form of the ignore pass (K4b-lean + K4b-exact): records whose filter leaves a (record, GT) pair undecided
  uint32_t* pend_queue;            // [B * n_img] global record ids (img * n_img + anchor_base[l] + rin)
  unsigned int* pend_count;        // number of queued records
  unsigned long long* obj_fixed;   // [3] object-loss terms of the queued records, 2^-32 fixed point (order-independent sum)
  double* partials;     // [n_cta]      object_loss partial of each ignore-kernel CTA
  double* partials_obj; // [3*B*YL_TERM_SPLIT,3] xy, wh, cls partials of each terms-kernel CTA (level-major)
};

__device__ __forceinline__ void yl_locate(const YlLevels& lv, int cta, int& l, int& img, int& chunk) {
  l = 0;
#pragma unroll
  for (int k = 1; k < YL_LEVELS; ++k) if (cta >= lv.cta_base[k]) l = k;
  const int r = cta - lv.cta_base[l];
  img = r / lv.chunks_per_img[l];
  chunk = r - img * lv.chunks_per_img[l];
}

// A box is "regular" when the cheap no-overlap reject is exact for it: finite, strictly positive extent and
// area, aspect term not NaN.  For two regular boxes  min(a2,b2)-max(a0,b0) <= 0  <=>  a2 <= b0 || b2 <= a0.
__device__ __forceinline__ bool yl_regular(const BoxT& b) {
  return (b.c2 > b.c0) && (b.c3 > b.c1) && (b.area > 0.0f) && (b.area < 3.0e38f) && (b.at == b.at) &&
         (dm_fabsf(b.c0) < 3.0e38f) && (dm_fabsf(b.c1) < 3.0e38f) && (dm_fabsf(b.c2) < 3.0e38f) && (dm_fabsf(b.c3) < 3.0e38f);
}

#define YL_OBJ_PER_THREAD 4
#define YL_OBJ_CHUNK (YL_CHUNK * YL_OBJ_PER_THREAD)

#define YL_SORT_CAP 2048
__device__ __forceinline__ void yl_gtprep_body(const YlParams& p, int l, int img, int* s_idx) {
  const int nthr = blockDim.x;
  const int rpi = p.lv.rec_per_img[l];
  const float* yt = p.sp_t ? nullptr : p.lv.y_true[l] + ((size_t)img * rpi) * p.RF;
  const int n = __ldcg(&p.gt_count[img * YL_LEVELS + l]);
  const size_t gbase = (size_t)img * p.n_img + p.lv.anchor_base[l];
  // The scan kernel appended the object records with atomics, i.e. in a run-dependent order; the xy / wh / class terms
  // are summed in list order (fp64, then one fp32 cast), so the list is put into ascending record order first: the
  // loss is then bit-reproducible run to run (lists longer than YL_SORT_CAP keep the atomic order).  The sparse-target
  // path builds its list in box order already.
  if (!p.sp_t && n > 1 && n <= YL_SORT_CAP) {
    for (int k = threadIdx.x; k < n; k += nthr) s_idx[k] = __ldcg(&p.obj_index[gbase + k]);
    __syncthreads();
    for (int k = threadIdx.x; k < n; k += nthr) {
      const int mine = s_idx[k];
      int rank = 0;
      for (int j = 0; j < n; ++j) rank += (s_idx[j] < mine) ? 1 : 0;  // record indices are unique
      p.obj_index[gbase + rank] = mine;
    }
    __syncthreads();
  }
  for (int k = threadIdx.x; k < n; k += nthr) {
    float tx, ty, tw, th;
    if (p.sp_t) {
      const float4 v = p.sp_t[gbase + k];
      tx = v.x; ty = v.y; tw = v.z; th = v.w;
    } else {
      const float* t = yt + (size_t)__ldcg(&p.obj_index[gbase + k]) * p.RF;
      tx = __ldg(t); ty = __ldg(t + 1); tw = __ldg(t + 2); th = __ldg(t + 3);
    }
    const float hx = DM_DIV(tw, 2.0f), hy = DM_DIV(th, 2.0f);
    BoxT g = bm_prep(DM_SUB(tx, hx), DM_SUB(ty, hy), DM_ADD(tx, hx), DM_ADD(ty, hy), p.metric);
    p.gt_box[gbase + k] = make_float4(g.c0, g.c1, g.c2, g.c3);
    p.gt_aux[gbase + k] = make_float4(g.area, g.at, dm_logf(g.area), yl_regular(g) ? 1.0f : 0.0f);
  }
}

__global__ void __launch_bounds__(128) yolo_loss_gtprep_kernel(YlParams p) {
  __shared__ int s_idx[YL_SORT_CAP];
  const int l = blockIdx.x / p.B;
  yl_gtprep_body(p, l, blockIdx.x - l * p.B, s_idx);
}

// K4a: pure stream over the obj channel.  Objects (obj != 0) are appended to the (image, level) object list in
// obj_index; their terms are computed by the next kernel, when the memory system is no longer saturated by the scan
// (doing it here cost a second DRAM round trip per CTA behind everyone else's scan loads: 42 us vs 30 + 4).
__global__ void __launch_bounds__(YL_CHUNK) yolo_loss_scan_kernel(YlParams p) {
  __shared__ int s_list[YL_OBJ_CHUNK];
  __shared__ int s_idx[YL_SORT_CAP];
  __shared__ int s_n, s_base;
  __shared__ bool s_last;
  // same (level, image, chunk) decomposition as the ignore kernel but with larger chunks.  The CTAs walk y_true from its
  // end: the part GetTargets wrote last is still in L2
  int l = 0;
  const int bid = (int)(gridDim.x - 1 - blockIdx.x);
#pragma unroll
  for (int k = 1; k < YL_LEVELS; ++k) if (bid >= p.lv.obj_cta_base[k]) l = k;
  const int rcta = bid - p.lv.obj_cta_base[l];
  const int img = rcta / p.lv.obj_chunks_per_img[l];
  const int chunk = rcta - img * p.lv.obj_chunks_per_img[l];
  const int rpi = p.lv.rec_per_img[l];
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  const float* yt = p.lv.y_true[l] + ((size_t)img * rpi) * p.RF;
  float objv[YL_OBJ_PER_THREAD];
#pragma unroll
  for (int u = 0; u < YL_OBJ_PER_THREAD; ++u) {  // independent strided sector reads, all in flight together
    const int rin = chunk * YL_OBJ_CHUNK + u * YL_CHUNK + (int)threadIdx.x;
    objv[u] = (rin < rpi) ? __ldcg(yt + (size_t)rin * p.RF + 4) : 0.0f;
  }
#pragma unroll
  for (int u = 0; u < YL_OBJ_PER_THREAD; ++u) {
    const int rin = chunk * YL_OBJ_CHUNK + u * YL_CHUNK + (int)threadIdx.x;
    if (rin < rpi) {
      p.obj_compact[(size_t)img * p.n_img + p.lv.anchor_base[l] + rin] = objv[u];
      if (objv[u] != 0.0f) s_list[atomicAdd(&s_n, 1)] = rin;
    }
  }
  __syncthreads();
  const int n = s_n;
  if (n > 0) {   // block-uniform
    if (threadIdx.x == 0) s_base = atomicAdd(&p.gt_count[img * YL_LEVELS + l], n);
    __syncthreads();
    int32_t* dst = p.obj_index + (size_t)img * p.n_img + p.lv.anchor_base[l] + s_base;
    for (int i = threadIdx.x; i < n; i += YL_CHUNK) dst[i] = s_list[i];
  }
  if (!p.scan_ticket) return;
  // K4a' without a launch: the last CTA of this (image, level) to finish prepares its GT list
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    s_last = atomicAdd(&p.scan_ticket[img * YL_LEVELS + l], 1u) == (unsigned)p.lv.obj_chunks_per_img[l] - 1u;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  yl_gtprep_body(p, l, img, s_idx);
}

// K4a': one thread per object: the prepared GT box of the ignore mask (corners of (t_xy, t_wh), tyu:68-71; area,
// atan(w/h), log area, "regular" flag).  One CTA per (level, image).
// A warp per object record: xy / wh / class terms (tyu:107-118).  Runs as the trailing 3*B*YL_TERM_SPLIT CTAs of the
// ignore kernel's grid (two dependent DRAM round trips and ~600 serial instructions per object: hidden under the
// ignore pass instead of sitting on the critical path).  CTA (l, img, s) takes objects k = s*4 + warp, stepping by
// 4*YL_TERM_SPLIT.
#define YL_TERM_SPLIT 16

__device__ __forceinline__ void yl_terms_body(const YlParams& p, int cta, double (*s_acc)[3]) {
  const int l = cta / (p.B * YL_TERM_SPLIT);
  const int rem = cta - l * (p.B * YL_TERM_SPLIT);
  const int img = rem / YL_TERM_SPLIT, split = rem - img * YL_TERM_SPLIT;
  const int rpi = p.lv.rec_per_img[l];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float* yt = p.sp_t ? nullptr : p.lv.y_true[l] + ((size_t)img * rpi) * p.RF;
  const float* yp = p.lv.y_pred[l] + ((size_t)img * rpi) * p.RF;
  const int n = p.gt_count[img * YL_LEVELS + l];
  const size_t gbase = (size_t)img * p.n_img + p.lv.anchor_base[l];
  double a_xy = 0.0, a_wh = 0.0, a_cls = 0.0;
  const int W = p.lv.w[l], H = p.lv.h[l];
  for (int k = split * (YL_ICHUNK / 32) + warp; k < n; k += YL_TERM_SPLIT * (YL_ICHUNK / 32)) {
    const int r = p.obj_index[gbase + k];
    const float* t = yt + (size_t)r * p.RF;
    const float* q = yp + (size_t)r * p.RF;
    float obj, tx, ty, tw, th;
    int sp_class = -1;
    if (p.sp_t) {  // the record the dense scatter would have written: obj = 1, one-hot class (cds:246-262)
      const float4 v = p.sp_t[gbase + k];
      obj = 1.0f; tx = v.x; ty = v.y; tw = v.z; th = v.w;
      sp_class = p.sp_cls[gbase + k];
    } else {
      obj = __ldg(t + 4);
      tx = __ldg(t); ty = __ldg(t + 1); tw = __ldg(t + 2); th = __ldg(t + 3);
    }
    const float scale = DM_SUB(2.0f, DM_MUL(tw, th));
    const float os = DM_MUL(obj, scale);  // (obj * scale) * term, evaluation order of tyu:109-110
    float e_xy = 0.f, e_wh = 0.f, e_cls = 0.f;
    if (lane < 2) {
      const int cell = r / p.A;
      const int gy = cell / W, gx = cell - gy * W;
      const float tv = lane == 0 ? tx : ty;
      const float g = lane == 0 ? (float)gx : (float)gy;
      const float gs = lane == 0 ? (float)W : (float)H;
      float raw = DM_SUB(DM_MUL(tv, gs), g);
      if (p.variant == YL_VARIANT_TF_YOLO_UTILS) raw = DM_MUL(obj, raw);  // tyu:44 (absent in yolo_loss.py:120)
      e_xy = DM_MUL(os, dm_bce_logits(raw, __ldg(q + lane)));
    } else if (lane < 4) {
      const int a = r - (r / p.A) * p.A;
      const float tv = lane == 2 ? tw : th;
      const float im = lane == 2 ? p.img_w : p.img_h;
      const float an = lane == 2 ? p.lv.anc_w[l][a] : p.lv.anc_h[l][a];
      float num = DM_MUL(tv, im);
      if (p.variant == YL_VARIANT_TF_YOLO_UTILS) num = DM_ADD(num, 1e-8f);  // tyu:48
      const float raw = dm_logf(DM_DIV(num, an));
      const float d = DM_SUB(raw, __ldg(q + lane));
      e_wh = DM_MUL(DM_MUL(os, 0.5f), DM_MUL(d, d));
    }
    if (p.sp_t) {
      for (int c = 5 + lane; c < p.RF; c += 32) e_cls += DM_MUL(obj, dm_bce_logits((c - 5 == sp_class) ? 1.0f : 0.0f, __ldg(q + c)));
    } else {
      for (int c = 5 + lane; c < p.RF; c += 32) e_cls += DM_MUL(obj, dm_bce_logits(__ldg(t + c), __ldg(q + c)));
    }
    e_xy = warp_sum(e_xy); e_wh = warp_sum(e_wh); e_cls = warp_sum(e_cls);
    if (lane == 0) { a_xy += (double)e_xy; a_wh += (double)e_wh; a_cls += (double)e_cls; }
  }
  if (lane == 0) { s_acc[warp][0] = a_xy; s_acc[warp][1] = a_wh; s_acc[warp][2] = a_cls; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double x = 0, w = 0, c = 0;
    for (int i = 0; i < YL_ICHUNK / 32; ++i) { x += s_acc[i][0]; w += s_acc[i][1]; c += s_acc[i][2]; }
    double* out = p.partials_obj + (size_t)cta * 3;
    out[0] = x; out[1] = w; out[2] = c;
  }
}

// Decode-free necessary conditions for metric(P,G) >= thr when thr >= 0.5 (DESIGN.md "ignore-mask filter"):
//  (a) every metric of the family is <= IoU <= min(area)/max(area)  =>  both areas within a factor thr of each
//      other; the predicted area is exp(tw+th)*anchor_area/image_area up to ~1 %, so this is a window on the
//      raw logit sum  s' = tw + th + log(anchor_area/image_area):  log(thr*Ag) - 0.05 <= s' <= log(Ag/thr) + 0.05;
//  (b) IoU >= 0.5 needs >= half of P's width and height inside G, so P's centre lies inside G; the centre is
//      (sigmoid(t)+grid)/grid_wh, i.e. inside the anchor's grid cell, so the cell rectangle (grown by 1e-3)
//      must intersect G.
// Both use only tw, th and the cell index; a lane decodes its box (2 sigmoid, 2 exp, atan) only when some GT
// passes both, and then runs the exact test.  Lanes with |t| outside [-6,4] or NaN, irregular GTs and thr < 0.5
// take the exact path against every GT.
#define YL_IOU_EPS 5e-3f
#define YL_IOU_FLOOR 1e-2f
#define YL_CELL_MARGIN 1e-3f
#define YL_LOG_MARGIN 0.05f

// BCE-with-logits for the (continuous) loss value only: MUFU-based exp/log, relative error ~1e-6 per term,
// far inside the 1e-4 loss tolerance; decisions never use it.
__device__ __forceinline__ float yl_fast_bce(float z, float x) {
  const float e = __expf(-fabsf(x));
  return fmaxf(x, 0.0f) - x * z + __logf(1.0f + e);
}

__device__ __forceinline__ int yl_fastdiv(int n, uint32_t magic) {
  return magic == 0u ? n : (int)__umulhi((uint32_t)n, magic);  // magic 0 encodes divisor 1
}

// obj of the record at flat anchor index `ain` of image `img`: one bit (sparse-target mode) or the scan's compact copy
__device__ __forceinline__ float yl_obj(const YlParams& p, int img, int ain) {
  if (p.obj_bits) return ((__ldg(p.obj_bits + (size_t)img * p.bits_words + (ain >> 5)) >> (ain & 31)) & 1u) ? 1.0f : 0.0f;
  return p.obj_compact[(size_t)img * p.n_img + ain];
}

// tx, ty, tw, th, conf of a record that starts sh = 0..3 floats into the 8 loaded floats (lo, hi): rotate them left by sh
// with two select stages
__device__ __forceinline__ void yl_rotate5(const float4 lo, const float4 hi, int sh, float& tx, float& ty, float& tw, float& th,
                                           float& pobj) {
  const bool s1 = sh & 1, s2 = sh & 2;
  const float a0 = s1 ? lo.y : lo.x, a1 = s1 ? lo.z : lo.y, a2 = s1 ? lo.w : lo.z, a3 = s1 ? hi.x : lo.w;
  const float a4 = s1 ? hi.y : hi.x, a5 = s1 ? hi.z : hi.y, a6 = s1 ? hi.w : hi.z;
  tx = s2 ? a2 : a0; ty = s2 ? a3 : a1; tw = s2 ? a4 : a2; th = s2 ? a5 : a3; pobj = s2 ? a6 : a4;
}

// One record's object_loss = obj*bce + (1-obj)*bce*ignore (tyu:114).  Also writes the record's ignore byte and
// d loss / d conf logit = (sigmoid(p) - obj) * (obj + (1-obj)*ignore) / B (the mask has no gradient).  `filtered`: the
// lean filter alone decided ignore = 1, and the gradient is taken as (sigmoid(p) - obj) / B.  The factor equals 1 in
// exact arithmetic but not always in fp32 for a non-binary obj, so each form keeps its own bits.
__device__ __forceinline__ float yl_record_term(const YlParams& p, int l, int img, int ain, float obj, float pobj, bool hit,
                                                bool filtered) {
  const float bc = yl_fast_bce(obj, pobj);
  const float ign = hit ? 0.0f : 1.0f;
  const float e = obj * bc + (1.0f - obj) * bc * ign;
  if (p.out_ignore) p.out_ignore[(size_t)img * p.n_img + ain] = hit ? 0 : 1;
  if (p.conf_grad) {
    const float ex = __expf(-fabsf(pobj));
    const float rr = 1.0f / (1.0f + ex);
    const float sg = pobj >= 0.0f ? rr : ex * rr;
    p.conf_grad[(size_t)p.B * p.lv.anchor_base[l] + (size_t)img * p.lv.rec_per_img[l] + (ain - p.lv.anchor_base[l])] =
        filtered ? (sg - obj) * p.inv_div : (sg - obj) * (obj + (1.0f - obj) * ign) * p.inv_div;
  }
  return e;
}

// The CTA's object-loss partial: an fp32 sum of each warp's 32 terms, fp64 across the warps (and across the CTAs in K4c)
__device__ __forceinline__ void yl_store_partial(const YlParams& p, int icta, float e, double* s_acc) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  e = warp_sum(e);
  if (lane == 0) s_acc[warp] = (double)e;
  __syncthreads();
  if (threadIdx.x == 0) {
    double sum = 0;
    for (int i = 0; i < YL_ICHUNK / 32; ++i) sum += s_acc[i];
    p.partials[icta] = sum;
  }
}

// The filter's per-record state, shared by both forms of the ignore pass.
struct YlFilter {
  bool nice;                         // logits in the range where the decode-free bounds are proven
  bool fast_ok;                      // the approximate box may decide the IoU reject
  bool any_rough;                    // some active lane of the warp is not nice: every GT is relevant
  float sp;                          // tw + th + log(anchor area / image area)
  float fx0, fy0, fx1, fy1, farea;   // approximate decoded box
  float cx0, cy0, cx1, cy1;          // rectangle that certainly contains the decoded centre
  float ux0, uy0, ux1, uy1;          // the warp's strip of cells
  float lo_k, hi_k, thr_lo;
};

// Every lane of the warp calls this (it shuffles); inactive lanes are never nice.
__device__ __forceinline__ YlFilter yl_filter_init(const YlParams& p, int l, int rin, bool active, float tx, float ty,
                                                   float tw, float th) {
  YlFilter f = {};
  const int W = p.lv.w[l], H = p.lv.h[l];
  const int cell = yl_fastdiv(rin, p.magic_a);
  const int a = min(rin - cell * p.A, 7);
  const int gy = yl_fastdiv(cell, p.lv.magic_w[l]);
  const int gx = cell - gy * W;
  const bool filter_ok = p.thr >= 0.5f;
  f.nice = active && filter_ok && (tw >= p.tmin_w[l][a]) && (tw <= 4.0f) && (th >= p.tmin_h[l][a]) && (th <= 4.0f) &&
           (tx == tx) && (ty == ty);
  f.sp = tw + th + p.logk[l][a];
  const float invW = 1.0f / (float)W, invH = 1.0f / (float)H;
  // (c) approximate decode (MUFU exp / reciprocal; corner error < 2e-6 for boxes up to 2 image widths) for an
  // IoU *upper-bound* reject: every metric of the family is <= IoU, so IoU_fast < thr - YL_IOU_EPS with both
  // overlap extents >= YL_IOU_FLOOR (relative IoU error then < 3.2e-3, DESIGN.md) proves metric < thr.  Accepts
  // are never decided here: pairs that survive go to the exact test.
  if (f.nice) {
    const float ex = __expf(-fabsf(tx)), ey = __expf(-fabsf(ty));
    const float rx = __fdividef(1.0f, 1.0f + ex), ry = __fdividef(1.0f, 1.0f + ey);
    const float fx = ((tx >= 0.0f ? rx : ex * rx) + (float)gx) * invW, fy = ((ty >= 0.0f ? ry : ey * ry) + (float)gy) * invH;
    const float fw = __expf(tw) * __fdividef(p.lv.anc_w[l][a], p.img_w), fh = __expf(th) * __fdividef(p.lv.anc_h[l][a], p.img_h);
    f.fx0 = fx - 0.5f * fw; f.fx1 = fx + 0.5f * fw; f.fy0 = fy - 0.5f * fh; f.fy1 = fy + 0.5f * fh;
    f.farea = fw * fh;
    f.fast_ok = (fw <= 2.0f) && (fh <= 2.0f);
  }
  f.thr_lo = p.thr - YL_IOU_EPS;
  f.cx0 = (float)gx * invW - YL_CELL_MARGIN; f.cx1 = (float)(gx + 1) * invW + YL_CELL_MARGIN;
  f.cy0 = (float)gy * invH - YL_CELL_MARGIN; f.cy1 = (float)(gy + 1) * invH + YL_CELL_MARGIN;
  // the warp's 32 consecutive records cover a run of cells: rows gy(first)..gy(last); one row -> x range of
  // the run, several rows -> full width.  (Superset of the nice lanes' cells: conservative.)
  const uint32_t act = __ballot_sync(0xffffffffu, active);
  if (act) {
    const int first = __ffs(act) - 1, last = 31 - __clz(act);
    const float first_x0 = __shfl_sync(0xffffffffu, f.cx0, first), first_y0 = __shfl_sync(0xffffffffu, f.cy0, first);
    const float last_x1 = __shfl_sync(0xffffffffu, f.cx1, last), last_y1 = __shfl_sync(0xffffffffu, f.cy1, last);
    const int gyf = __shfl_sync(0xffffffffu, gy, first), gyl = __shfl_sync(0xffffffffu, gy, last);
    f.uy0 = first_y0; f.uy1 = last_y1;
    f.ux0 = (gyf == gyl) ? first_x0 : -1.0f;
    f.ux1 = (gyf == gyl) ? last_x1 : 2.0f;
  }
  f.any_rough = __any_sync(0xffffffffu, active && !f.nice);
  f.lo_k = p.log_thr - YL_LOG_MARGIN; f.hi_k = -p.log_thr + YL_LOG_MARGIN;
  return f;
}

// The filter proves metric < thr for this lane's record and the prepared GT (corners c; area, atan term, log area,
// regular flag x).  All rejects as straight-line predicate arithmetic (bitwise, no short-circuit branches): the warp
// executes the tests of every relevant GT anyway, and the divergence bookkeeping of early exits cost more than it saved.
__device__ __forceinline__ bool yl_pair_rejected(const YlFilter& f, const float4 c, const float4 x) {
  const float iw = fminf(f.fx1, c.z) - fmaxf(f.fx0, c.x), ih = fminf(f.fy1, c.w) - fmaxf(f.fy0, c.y);
  const float inter = iw * ih;
  const bool cell_rej = (f.cx1 < c.x) | (c.z < f.cx0) | (f.cy1 < c.y) | (c.w < f.cy0);
  const bool win_rej = (f.sp < x.z + f.lo_k) | (f.sp > x.z + f.hi_k);
  const bool dis_rej = (iw < -1e-5f) | (ih < -1e-5f);  // disjoint by far more than the decode error
  const bool iou_rej = f.fast_ok & (iw >= YL_IOU_FLOOR) & (ih >= YL_IOU_FLOOR) & (inter < f.thr_lo * (f.farea + x.x - inter));
  return f.nice & (x.w != 0.0f) & (cell_rej | win_rej | dis_rej | iou_rej);
}

// visit(g, c, x, rejected) for every GT g of the list that can touch the warp's strip of cells, in ascending order;
// irregular GTs (x.w == 0) and warps with rough lanes take every GT.  The whole warp walks the same GTs.
template <class Visit>
__device__ __forceinline__ void yl_filter_gts(const YlFilter& f, const float4* gbox, const float4* gaux, int n_gt, Visit&& visit) {
  const int lane = threadIdx.x & 31;
  for (int j0 = 0; j0 < n_gt; j0 += 32) {
    const int j = j0 + lane;
    bool relevant = false;
    if (j < n_gt) {
      const float4 c = __ldg(gbox + j);
      relevant = f.any_rough || (__ldg(gaux + j).w == 0.0f) || !((f.ux1 < c.x) || (c.z < f.ux0) || (f.uy1 < c.y) || (c.w < f.uy0));
    }
    uint32_t mask = __ballot_sync(0xffffffffu, relevant);
    while (mask) {
      const int g = j0 + __ffs(mask) - 1;
      mask &= mask - 1u;
      const float4 c = __ldg(gbox + g);
      const float4 x = __ldg(gaux + g);
      visit(g, c, x, yl_pair_rejected(f, c, x));
    }
  }
}

// Three phases per CTA of YL_ICHUNK (128) records:
//  1. (all lanes, decode-free) each record tests the GTs that can touch its warp's strip of grid cells with the
//     cell / logit-sum windows and pushes surviving (record, gt) pairs to a shared-memory queue;
//  2. (dense) the queue is drained with one pair per thread: exact decode of the record (2 sigmoid, 2 exp, atan),
//     exact overlap / area tests and the exact metric — the expensive arithmetic runs at full lane utilisation
//     and only for pairs that need it;
//  3. object_loss = obj*bce + (1-obj)*bce*ignore for every record.
// The GT list is read straight from global memory (packed float4 pairs, L1-resident).
#define YL_QCAP 1024
#define YL_IMINB 8   // 64 registers: no spills; 10 (48 registers) spills and is 5 us slower

// exact decode of a record (tyu:57,61: xy = (sigmoid(t)+grid)/grid_wh ; wh = exp(t)*anchor/image_wh, no inf guard, Q7)
__device__ __forceinline__ BoxT yl_decode_record(const YlParams& p, int l, int rin, float tx, float ty, float tw, float th) {
  const int W = p.lv.w[l], H = p.lv.h[l];
  const int cell = yl_fastdiv(rin, p.magic_a);
  const int a = min(rin - cell * p.A, 7);
  const int gy = yl_fastdiv(cell, p.lv.magic_w[l]);
  const int gx = cell - gy * W;
  const float x_ = DM_DIV(DM_ADD(dm_sigmoidf(tx), (float)gx), (float)W);
  const float y_ = DM_DIV(DM_ADD(dm_sigmoidf(ty), (float)gy), (float)H);
  const float w_ = DM_DIV(DM_MUL(dm_expf(tw), p.lv.anc_w[l][a]), p.img_w);
  const float h_ = DM_DIV(DM_MUL(dm_expf(th), p.lv.anc_h[l][a]), p.img_h);
  const float hx_ = DM_DIV(w_, 2.0f), hy_ = DM_DIV(h_, 2.0f);
  return bm_prep(DM_SUB(x_, hx_), DM_SUB(y_, hy_), DM_ADD(x_, hx_), DM_ADD(y_, hy_), B200_METRIC_YOLO_IOU);
}

// exact test of a decoded record against one prepared ground-truth box (c = corners, x = area, atan term, log area,
// regular flag): metric >= thr, or NaN (tf.reduce_max propagates NaN and NaN < thr is False)
__device__ __forceinline__ bool yl_box_hits(const YlParams& p, BoxT pb, bool pb_regular, const float4 c, const float4 x) {
  BoxT gb; gb.c0 = c.x; gb.c1 = c.y; gb.c2 = c.z; gb.c3 = c.w; gb.area = x.x; gb.at = x.y;
  if (x.w != 0.0f && p.thr > 0.0f && pb_regular) {
    // exact rejects for regular pairs: no overlap, or areas further apart than thr allows (iou <= min/max)
    if ((pb.c2 <= c.x) || (c.z <= pb.c0) || (pb.c3 <= c.y) || (c.w <= pb.c1)) return false;
    if (fminf(pb.area, x.x) < 0.99f * p.thr * fmaxf(pb.area, x.x)) return false;
  }
  if (p.metric == B200_METRIC_YOLO_CIOU) pb.at = dm_atanf(DM_DIV(DM_SUB(pb.c2, pb.c0), DM_SUB(pb.c3, pb.c1)));
  if (bm_surely_below(pb, gb, p.metric, p.thr)) return false;
  const float mm = bm_metric(pb, gb, p.metric);
  return (mm >= p.thr) || (mm != mm);
}

__device__ __forceinline__ bool yl_pair_hits(const YlParams& p, int l, int rin, float tx, float ty, float tw, float th,
                                             const float4 c, const float4 x) {
  const BoxT pb = yl_decode_record(p, l, rin, tx, ty, tw, th);
  return yl_box_hits(p, pb, yl_regular(pb), c, x);
}

// The single-kernel form.  Where a level is 16-byte aligned and a record holds at least 8 floats, two neighbouring lanes
// fetch the five logits of a record with one request (see the load section): what bounds the kernel when y_pred is read
// in place from pinned host memory over PCIe.  Other levels load the five floats one by one.
__global__ void __launch_bounds__(YL_ICHUNK, YL_IMINB) yolo_loss_ignore_kernel(YlParams p) {
  __shared__ float4 s_t[YL_ICHUNK];
  __shared__ uint32_t s_q[YL_QCAP];
  __shared__ uint32_t s_hit[YL_ICHUNK / 32];
  __shared__ int s_nq;
  __shared__ double s_acc[YL_ICHUNK / 32];
  const int n_term_cta = YL_LEVELS * p.B * YL_TERM_SPLIT;
  const int n_icta = (int)gridDim.x - n_term_cta;
  if ((int)blockIdx.x >= n_icta) {  // block-uniform
    __shared__ double s_tacc[YL_ICHUNK / 32][3];
    yl_terms_body(p, blockIdx.x - n_icta, s_tacc);
    return;
  }
  const int icta = blockIdx.x;
  int l, img, chunk;
  yl_locate(p.lv, icta, l, img, chunk);
  const int rpi = p.lv.rec_per_img[l];
  const int rin = chunk * YL_ICHUNK + (int)threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool active = rin < rpi;
  const int n_gt = p.gt_count[img * YL_LEVELS + l];
  const float4* gbox = p.gt_box + (size_t)img * p.n_img + p.lv.anchor_base[l];
  const float4* gaux = p.gt_aux + (size_t)img * p.n_img + p.lv.anchor_base[l];
  float obj = 0.f, tx = 0.f, ty = 0.f, tw = 0.f, th = 0.f, pobj = 0.f;
  // block-uniform.  The two aligned 16-byte loads cover floats [f0 & ~3, (f0 & ~3) + 8): inside the tensor only when a
  // record holds at least 8 floats (C >= 3); narrower records take the scalar path
  const bool aligned = ((reinterpret_cast<uintptr_t>(p.lv.y_pred[l]) & 15) == 0) && (p.RF >= 8);
  if (active) obj = yl_obj(p, img, p.lv.anchor_base[l] + rin);
  if (aligned) {
    // tx,ty,tw,th,conf of a record sit at float offset f0; the two aligned 16-byte chunks that cover them are fetched
    // by two neighbouring lanes of ONE load instruction (16 records per instruction, two instructions per warp), so a
    // record costs one memory request (one 128-byte line, 1-2 sectors) instead of two — this halves the request count,
    // which is what bounds the kernel when y_pred is read in place from pinned host memory over PCIe
    const float4* base = reinterpret_cast<const float4*>(p.lv.y_pred[l]);
    const int sub = lane & 1, rsel = lane >> 1;
    float4 ld[2];
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const int rin_t = chunk * YL_ICHUNK + warp * 32 + 16 * t + rsel;
      ld[t] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (rin_t < rpi) ld[t] = __ldcg(base + ((((size_t)img * rpi + rin_t) * p.RF) >> 2) + sub);
    }
    // lane r takes the pair loaded by lanes 2(r mod 16), 2(r mod 16)+1 of instruction r / 16
    const int src = (lane & 15) << 1;
    auto take = [&](int from) {
      float4 v[2];
#pragma unroll
      for (int t = 0; t < 2; ++t)
        v[t] = make_float4(__shfl_sync(0xffffffffu, ld[t].x, from), __shfl_sync(0xffffffffu, ld[t].y, from),
                           __shfl_sync(0xffffffffu, ld[t].z, from), __shfl_sync(0xffffffffu, ld[t].w, from));
      return lane >= 16 ? v[1] : v[0];
    };
    const float4 lo = take(src), hi = take(src + 1);
    if (active) yl_rotate5(lo, hi, (int)((((size_t)img * rpi + rin) * p.RF) & 3), tx, ty, tw, th, pobj);
  } else if (active) {
    const float* q = p.lv.y_pred[l] + ((size_t)img * rpi + rin) * p.RF;
    tx = __ldcg(q); ty = __ldcg(q + 1); tw = __ldcg(q + 2); th = __ldcg(q + 3); pobj = __ldcg(q + 4);
  }
  bool hit = false;  // some GT with metric >= thr (or NaN)
  if (n_gt > 0) {    // block-uniform
    if (threadIdx.x == 0) s_nq = 0;
    if (threadIdx.x < YL_ICHUNK / 32) s_hit[threadIdx.x] = 0u;
    s_t[threadIdx.x] = make_float4(tx, ty, tw, th);
    __syncthreads();
    // ---------------- phase 1 ----------------
    const YlFilter f = yl_filter_init(p, l, rin, active, tx, ty, tw, th);
    yl_filter_gts(f, gbox, gaux, n_gt, [&](int g, const float4 c, const float4 x, bool rejected) {
      if (!active | hit | rejected) return;
      const int slot = atomicAdd(&s_nq, 1);
      if (slot < YL_QCAP) s_q[slot] = (threadIdx.x << 24) | (uint32_t)g;            // drained in phase 2
      else {  // queue full: exact test now.  The logits pass through an opaque asm so that the compiler cannot
              // hoist the record decode in front of the filter loop (it did: ~200 instructions per warp, always).
        float otx = tx, oty = ty, otw = tw, oth = th;
        asm volatile("" : "+f"(otx), "+f"(oty), "+f"(otw), "+f"(oth));
        if (yl_pair_hits(p, l, rin, otx, oty, otw, oth, c, x)) hit = true;
      }
    });
    if (hit) atomicOr(&s_hit[warp], 1u << lane);
    __syncthreads();
    // ---------------- phase 2 ----------------
    const int nq = min(s_nq, YL_QCAP);
    for (int q = threadIdx.x; q < nq; q += YL_ICHUNK) {
      const uint32_t e = s_q[q];
      const int r = (int)(e >> 24), g = (int)(e & 0xffffffu);
      if ((s_hit[r >> 5] >> (r & 31)) & 1u) continue;  // already decided (benign race: only skips work)
      const float4 t = s_t[r];
      if (yl_pair_hits(p, l, chunk * YL_ICHUNK + r, t.x, t.y, t.z, t.w, __ldg(gbox + g), __ldg(gaux + g)))
        atomicOr(&s_hit[r >> 5], 1u << (r & 31));
    }
    __syncthreads();
    hit = (s_hit[warp] >> lane) & 1u;
  }
  // ---------------- phase 3 ----------------
  float e = 0.f;
  if (active) e = yl_record_term(p, l, img, p.lv.anchor_base[l] + rin, obj, pobj, hit, false);
  yl_store_partial(p, icta, e, s_acc);
}

// ---- split form of K4b: device-resident y_pred, every level 16-byte aligned, records of >= 8 floats ----------------
// The filter of K4b rejects all but a few thousand (record, GT) pairs per batch; the exact decode + exact metric those few
// need is what makes K4b a 64-register kernel (8 CTAs per SM, ~45 % of the warp slots).  Here the stream is split:
//   K4b-lean   two aligned 16-byte loads per record, the same decode-free / approximate-IoU rejects (the filter helpers
//              above), BCE of every DECIDED record (no surviving pair => ignore = 1); a record with a surviving pair is
//              only queued (one global id per record).  No shared-memory queue, no exact code: far fewer registers, no
//              mid-kernel CTA barriers.
//   K4b-exact  a warp per queued record: the exact test (yl_pair_hits, with its own exact rejects) against EVERY ground
//              truth of the record's (image, level), lanes <-> GTs; writes the record's ignore bit / gradient and adds its
//              object-loss term to a 2^-32 fixed-point accumulator (integer atomics: the sum is order independent, so
//              the loss stays bit-reproducible).
// A rejected pair is provably below the threshold (DESIGN.md section 6), so "some surviving pair hits" == "some GT hits":
// the ignore mask is bit-identical to K4b's.
#define YL_FIXED_ONE 4294967296.0  // 2^32

// 10 CTAs per SM (48 registers, no spills): the fastest headline step of 8, 10, 12 and 16 (profiles/r02_ab_measurements.txt)
__global__ void __launch_bounds__(YL_ICHUNK, 10) yolo_loss_ignore_lean_kernel(YlParams p) {
  __shared__ double s_acc[YL_ICHUNK / 32];
  const int n_term_cta = YL_LEVELS * p.B * YL_TERM_SPLIT;
  const int n_icta = (int)gridDim.x - n_term_cta;
  if ((int)blockIdx.x >= n_icta) {  // block-uniform
    __shared__ double s_tacc[YL_ICHUNK / 32][3];
    yl_terms_body(p, blockIdx.x - n_icta, s_tacc);
    return;
  }
  const int icta = blockIdx.x;
  int l, img, chunk;
  yl_locate(p.lv, icta, l, img, chunk);
  const int rpi = p.lv.rec_per_img[l];
  const int rin = chunk * YL_ICHUNK + (int)threadIdx.x;
  const int lane = threadIdx.x & 31;
  const bool active = rin < rpi;
  const int n_gt = p.gt_count[img * YL_LEVELS + l];
  const float4* gbox = p.gt_box + (size_t)img * p.n_img + p.lv.anchor_base[l];
  const float4* gaux = p.gt_aux + (size_t)img * p.n_img + p.lv.anchor_base[l];
  float obj = 0.f, tx = 0.f, ty = 0.f, tw = 0.f, th = 0.f, pobj = 0.f;
  if (active) {
    obj = yl_obj(p, img, p.lv.anchor_base[l] + rin);
    // tx,ty,tw,th,conf sit at float offset f0; two aligned 16-byte loads cover them (L1 bypass)
    const size_t f0 = ((size_t)img * rpi + rin) * p.RF;
    const float4 lo = __ldcg(reinterpret_cast<const float4*>(p.lv.y_pred[l]) + (f0 >> 2));
    const float4 hi = __ldcg(reinterpret_cast<const float4*>(p.lv.y_pred[l]) + (f0 >> 2) + 1);
    yl_rotate5(lo, hi, (int)(f0 & 3), tx, ty, tw, th, pobj);
  }
  bool pending = false;  // some (record, GT) pair survives the rejects: K4b-exact decides
  if (n_gt > 0) {        // block-uniform
    const YlFilter f = yl_filter_init(p, l, rin, active, tx, ty, tw, th);
    yl_filter_gts(f, gbox, gaux, n_gt, [&](int, const float4, const float4, bool rejected) { pending |= active & !rejected; });
  }
  // queue the undecided records (warp-aggregated append), account for the decided ones
  {
    const uint32_t pm = __ballot_sync(0xffffffffu, pending);
    if (pm) {
      unsigned int base = 0;
      if (lane == 0) base = atomicAdd(p.pend_count, (unsigned int)__popc(pm));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (pending) p.pend_queue[base + __popc(pm & ((1u << lane) - 1u))] = (uint32_t)((size_t)img * p.n_img + p.lv.anchor_base[l] + rin);
    }
  }
  float e = 0.f;
  if (active && !pending) e = yl_record_term(p, l, img, p.lv.anchor_base[l] + rin, obj, pobj, false, true);
  yl_store_partial(p, icta, e, s_acc);
}

// the exact pass over the queued records: HALF a warp per record (two records in flight per warp: the pass is a chain of
// dependent loads per record — queue entry, record, GT list — so it is bound by how many records are in flight, not by
// lanes: an (image, level) has ~17 GTs on average, one or two rounds of 16), `gwarp` of `nwarps` warps
__device__ __forceinline__ void yl_exact_pass(const YlParams& p, unsigned int gwarp, unsigned int nwarps) {
  const int lane = threadIdx.x & 31;
  const int half = lane >> 4, sub = lane & 15;
  const unsigned int n = *p.pend_count;
  for (unsigned int q0 = gwarp * 2u; q0 < n; q0 += nwarps * 2u) {   // warp-uniform trip count
    const unsigned int q = q0 + (unsigned int)half;
    const bool valid = q < n;
    const uint32_t id = valid ? p.pend_queue[q] : 0u;
    const int img = (int)(id / (uint32_t)p.n_img);
    const int ain = (int)(id - (uint32_t)img * (uint32_t)p.n_img);
    int l = 0;
#pragma unroll
    for (int k = 1; k < YL_LEVELS; ++k) if (ain >= p.lv.anchor_base[k]) l = k;
    const int rin = ain - p.lv.anchor_base[l];
    const int rpi = p.lv.rec_per_img[l];
    const float* rec = p.lv.y_pred[l] + ((size_t)img * rpi + rin) * p.RF;
    const float tx = __ldg(rec), ty = __ldg(rec + 1), tw = __ldg(rec + 2), th = __ldg(rec + 3), pobj = __ldg(rec + 4);
    const float obj = yl_obj(p, img, ain);
    const int n_gt = valid ? p.gt_count[img * YL_LEVELS + l] : 0;
    const float4* gbox = p.gt_box + (size_t)img * p.n_img + p.lv.anchor_base[l];
    const float4* gaux = p.gt_aux + (size_t)img * p.n_img + p.lv.anchor_base[l];
    // the record is decoded once (every lane of the half the same values), then lanes <-> ground-truth boxes: the exact
    // no-overlap / area-ratio rejects dispose of almost all of them before a metric is evaluated
    const BoxT pb = yl_decode_record(p, l, rin, tx, ty, tw, th);
    const bool pb_regular = yl_regular(pb);
    bool hit = false;
    for (int g0 = 0;; g0 += 16) {
      const bool more = g0 < n_gt && !hit;
      if (!__any_sync(0xffffffffu, more)) break;
      const int g = g0 + sub;
      bool h = false;
      if (more && g < n_gt) h = yl_box_hits(p, pb, pb_regular, __ldg(gbox + g), __ldg(gaux + g));
      const uint32_t bal = __ballot_sync(0xffffffffu, h);
      hit = hit || ((bal >> (16 * half)) & 0xffffu) != 0u;
    }
    if (valid && sub == 0) {
      const float e = yl_record_term(p, l, img, ain, obj, pobj, hit, false);
      // non-finite terms (NaN / inf logits) cannot be carried in fixed point: they poison the sum through the top bit pattern
      if (e == e && e < 1.0e9f) atomicAdd(p.obj_fixed + l, (unsigned long long)((double)e * YL_FIXED_ONE + 0.5));
      else atomicOr(p.obj_fixed + l, 0x8000000000000000ull);
    }
  }
}

__global__ void __launch_bounds__(128) yolo_loss_ignore_exact_kernel(YlParams p) {
  yl_exact_pass(p, blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), gridDim.x * (blockDim.x >> 5));
}

// K4c: YL_FIN_CTAS CTAs each reduce an interleaved share of the per-CTA partials in fp64 (fixed assignment, fixed
// order); the CTA that takes the last ticket adds the YL_FIN_CTAS slices in index order and writes parts / loss.
// Deterministic run to run, and shorter than a single CTA walking all partials (shapes measured in DESIGN.md section 9).
#define YL_FIN_CTAS 32
#define YL_FIN_THREADS 256

struct YlFinalize {
  const double* partials; const double* partials_obj;
  int cta_base[YL_LEVELS + 1]; int obj_cta_base[YL_LEVELS + 1];
  float batch_divisor; float* parts; float* loss;
  double* slices;          // [YL_FIN_CTAS][12]
  unsigned int* ticket;    // zero on entry; reset by the last CTA
  B200Exchange xchg;       // data parallel: the 12 terms are summed over the ranks inside this kernel (world 1: no-op)
  const unsigned long long* obj_fixed;  // [3] or null: object-loss terms of the records K4b-exact decided (2^-32 fixed point)
  int publish_only;        // 1: store this rank's terms into the peers' mailboxes and return (b200_yolo_loss_collect_peer finishes)
};

// With `exact` (split form of the ignore pass) the launch is wider than YL_FIN_CTAS: every CTA first resolves its share of
// the queued records (K4b-exact inside this launch: no third kernel on the step's critical path), the first YL_FIN_CTAS
// CTAs also reduce their slices, and the ticket counts ALL CTAs.
__global__ void __launch_bounds__(YL_FIN_THREADS) yolo_loss_finalize_kernel(YlFinalize f, YlParams p, int exact) {
  __shared__ double s_red[YL_FIN_THREADS / 32][12];
  __shared__ bool s_last;
  if (exact) yl_exact_pass(p, blockIdx.x * (YL_FIN_THREADS / 32) + (threadIdx.x >> 5), gridDim.x * (YL_FIN_THREADS / 32));
  if ((int)blockIdx.x >= YL_FIN_CTAS) {   // block-uniform: exact-pass-only CTAs just take a ticket
    __syncthreads();
    if (threadIdx.x == 0) { __threadfence(); s_last = (atomicAdd(f.ticket, 1u) == gridDim.x - 1); }
    __syncthreads();
    if (!s_last) return;
  } else {
  double acc[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) acc[i] = 0.0;
  const int t0 = blockIdx.x * YL_FIN_THREADS + (int)threadIdx.x, stride = YL_FIN_CTAS * YL_FIN_THREADS;
#pragma unroll
  for (int l = 0; l < 3; ++l) {
#pragma unroll 4
    for (int c = f.cta_base[l] + t0; c < f.cta_base[l + 1]; c += stride) acc[l * 4 + 2] += f.partials[c];
    for (int c = f.obj_cta_base[l] + t0; c < f.obj_cta_base[l + 1]; c += stride) {
      acc[l * 4 + 0] += f.partials_obj[(size_t)c * 3 + 0];
      acc[l * 4 + 1] += f.partials_obj[(size_t)c * 3 + 1];
      acc[l * 4 + 3] += f.partials_obj[(size_t)c * 3 + 2];
    }
  }
  const int lane_ = threadIdx.x & 31, warp_ = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 12; ++i) {
    double v = warp_sum_d(acc[i]);
    if (lane_ == 0) s_red[warp_][i] = v;
  }
  __syncthreads();
  if (threadIdx.x < 12) {
    double s = 0.0;
    for (int w = 0; w < YL_FIN_THREADS / 32; ++w) s += s_red[w][threadIdx.x];
    f.slices[blockIdx.x * 12 + threadIdx.x] = s;
    __threadfence();
  }
  __syncthreads();
  if (threadIdx.x == 0) { __threadfence(); s_last = (atomicAdd(f.ticket, 1u) == gridDim.x - 1); }
  __syncthreads();
  if (!s_last) return;
  }
  __threadfence();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (warp == 0) {
    float v = 0.0f;
    if (lane < 12) {
      double s = 0.0;
      for (int g = 0; g < YL_FIN_CTAS; ++g) s += __ldcg(f.slices + g * 12 + lane);
      if (f.obj_fixed && (lane & 3) == 2) {
        const unsigned long long fx = __ldcg(f.obj_fixed + (lane >> 2));
        s += (fx >> 63) ? (double)__longlong_as_double(0x7ff8000000000000ll) : (double)fx * (1.0 / YL_FIXED_ONE);   // top bit = a non-finite term
      }
      v = DM_DIV((float)s, f.batch_divisor);  // reduce_sum(...) / batch_size_float, tyu:120-123
    }
    // data parallel (SURVEY 8e): batch_divisor is the GLOBAL batch, so the per-rank terms simply add up; the sum runs over
    // NVLink peer stores inside this warp, in rank order on every rank (exchange.cuh)
    if (f.publish_only && f.xchg.world > 1) xchg_publish_warp<float>(f.xchg, v, 12);
    else v = xchg_allreduce_warp<float>(f.xchg, v, 12);
    if (lane < 12 && f.parts) f.parts[lane] = v;
    float total = 0.0f;
    for (int l = 0; l < 3; ++l) {
      const float t0_ = __shfl_sync(0xffffffffu, v, l * 4 + 0), t1 = __shfl_sync(0xffffffffu, v, l * 4 + 1);
      const float t2 = __shfl_sync(0xffffffffu, v, l * 4 + 2), t3 = __shfl_sync(0xffffffffu, v, l * 4 + 3);
      total = DM_ADD(total, DM_ADD(DM_ADD(DM_ADD(t0_, t1), t2), t3));  // tyu:125
    }
    if (lane == 0) { *f.loss = total; *f.ticket = 0u; }
  }
}

// ---- backward: d loss / d y_pred (SURVEY §8f N1) ----------------------------------------------------------
// GetLoss is differentiated by tf.GradientTape in train_step (yolo_v4/model.py:318-338).  With BCE-with-logits
// d/dx = sigmoid(x) - z, and no gradient through the targets or the (boolean) ignore mask:
//   d/dt_xy  = obj*scale*(sigmoid(t) - raw_xy)/B      d/dt_wh = obj*scale*(t - raw_wh)/B
//   d/dconf  = (sigmoid(p) - obj)*(obj + (1-obj)*ignore)/B      d/dcls = obj*(sigmoid(c) - t_cls)/B
// The gradient tensor is dense like y_pred (7.7 MB/image at 608x608) but only the conf channel of every record and
// the full record of object cells are non-zero: one streaming write pass (conf values saved by the forward ignore
// kernel, 4 bytes/record) plus one warp per object record.
struct YlGradDense {
  float* grad[YL_LEVELS];
  const float* conf_grad[YL_LEVELS];
  unsigned long long quads[YL_LEVELS];     // cumulative number of 4-record groups per level
  unsigned long long records[YL_LEVELS];   // records per level (the last records % 4 are written by scalar stores)
  int RF;
};

// Four records = RF float4, always 16-byte aligned: a warp writes one such group per iteration (ceil(RF/32) 16-byte
// stores per lane), all zeros except the four conf channels, whose values are fetched by lanes 0-3 beforehand.  No
// index division, no load -> store dependency on the streaming path.
__global__ void __launch_bounds__(256) yolo_loss_grad_dense_kernel(YlGradDense g) {
  const int lane = threadIdx.x & 31;
  const unsigned long long total = g.quads[YL_LEVELS - 1];
  const unsigned long long wstride = (unsigned long long)gridDim.x * (blockDim.x >> 5);
  const int RF = g.RF;
  for (unsigned long long w = (unsigned long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); w < total; w += wstride) {
    // explicit selects: indexing the kernel-parameter arrays with a runtime level would copy them to local memory
    unsigned long long q = w;
    const float* cg = g.conf_grad[0];
    float* gr = g.grad[0];
    if (w >= g.quads[1]) { q = w - g.quads[1]; cg = g.conf_grad[2]; gr = g.grad[2]; }
    else if (w >= g.quads[0]) { q = w - g.quads[0]; cg = g.conf_grad[1]; gr = g.grad[1]; }
    const float mine = (lane < 4) ? __ldg(cg + q * 4ull + lane) : 0.0f;
    const float c0 = __shfl_sync(0xffffffffu, mine, 0), c1 = __shfl_sync(0xffffffffu, mine, 1);
    const float c2 = __shfl_sync(0xffffffffu, mine, 2), c3 = __shfl_sync(0xffffffffu, mine, 3);
    float4* dst = reinterpret_cast<float4*>(gr) + q * (unsigned long long)RF;
    for (int j = lane; j < RF; j += 32) {
      // float4 j of the group holds elements 4j..4j+3; record r's conf channel is element r*RF + 4
      const int e = 4 * j;
      float v[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int x = e + k - 4;  // == r*RF for the conf channel of record r
        v[k] = (x == 0) ? c0 : (x == RF) ? c1 : (x == 2 * RF) ? c2 : (x == 3 * RF) ? c3 : 0.0f;
      }
      __stcs(dst + j, make_float4(v[0], v[1], v[2], v[3]));
    }
  }
  // records beyond the last whole group of each level: scalar stores
  if (blockIdx.x == 0) {
#pragma unroll
    for (int l = 0; l < YL_LEVELS; ++l) {
      const unsigned long long r0 = g.records[l] & ~3ull, n_tail = (g.records[l] - r0) * (unsigned long long)RF;
      for (unsigned long long t = threadIdx.x; t < n_tail; t += blockDim.x) {
        const unsigned long long rec = r0 + t / (unsigned long long)RF;
        const int c = (int)(t % (unsigned long long)RF);
        g.grad[l][r0 * (unsigned long long)RF + t] = (c == 4) ? g.conf_grad[l][rec] : 0.0f;
      }
    }
  }
}

// YL_GRAD_SPLIT CTAs per (image, level): a warp per object record overwrites channels 0-3 and 5.. of that record
// (each object is two dependent DRAM round trips and ~85 sigmoids: spread wide instead of looping in one CTA).
// kSparse (b200_yolo_loss_from_boxes_grad): the targets of object slot k come from sp_t / sp_cls, i.e. the record the
// dense scatter would have written (obj = 1, one-hot class row; an out-of-range class id gives an all-zero row, as
// tf.one_hot); the arithmetic is the dense form's.
#define YL_GRAD_SPLIT 8
template <bool kSparse>
__global__ void __launch_bounds__(256) yolo_loss_grad_objects_kernel(YlParams p, float* g0, float* g1, float* g2) {
  const int pair = blockIdx.x / YL_GRAD_SPLIT, split = blockIdx.x - pair * YL_GRAD_SPLIT;
  const int img = pair / YL_LEVELS, l = pair - img * YL_LEVELS;
  float* grad = (l == 0 ? g0 : l == 1 ? g1 : g2);
  const int n = p.gt_count[img * YL_LEVELS + l];
  const int rpi = p.lv.rec_per_img[l];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int W = p.lv.w[l], H = p.lv.h[l];
  const float* yt = kSparse ? nullptr : p.lv.y_true[l] + ((size_t)img * rpi) * p.RF;
  const float* yp = p.lv.y_pred[l] + ((size_t)img * rpi) * p.RF;
  float* gr = grad + ((size_t)img * rpi) * p.RF;
  for (int k = split * 8 + warp; k < n; k += 8 * YL_GRAD_SPLIT) {
    const size_t slot = (size_t)img * p.n_img + p.lv.anchor_base[l] + k;
    const int r = p.obj_index[slot];
    const float* t = kSparse ? nullptr : yt + (size_t)r * p.RF;
    const float* q = yp + (size_t)r * p.RF;
    float* o = gr + (size_t)r * p.RF;
    float obj, tx, ty, tw, th;
    int sp_class = -1;
    if (kSparse) {
      const float4 v = p.sp_t[slot];
      obj = 1.0f; tx = v.x; ty = v.y; tw = v.z; th = v.w;
      sp_class = p.sp_cls[slot];
    } else {
      obj = __ldg(t + 4);
      tx = __ldg(t); ty = __ldg(t + 1); tw = __ldg(t + 2); th = __ldg(t + 3);
    }
    const float os = (obj * (2.0f - tw * th)) * p.inv_div;
    if (lane < 2) {
      const int cell = r / p.A;
      const int gy = cell / W, gx = cell - gy * W;
      float raw = (lane == 0 ? tx * (float)W - (float)gx : ty * (float)H - (float)gy);
      if (p.variant == YL_VARIANT_TF_YOLO_UTILS) raw = obj * raw;
      o[lane] = os * (dm_sigmoidf(__ldg(q + lane)) - raw);
    } else if (lane < 4) {
      const int a = r - (r / p.A) * p.A;
      float num = (lane == 2 ? tw * p.img_w : th * p.img_h);
      if (p.variant == YL_VARIANT_TF_YOLO_UTILS) num += 1e-8f;
      const float raw = dm_logf(num / (lane == 2 ? p.lv.anc_w[l][a] : p.lv.anc_h[l][a]));
      o[lane] = os * (__ldg(q + lane) - raw);
    }
    for (int c = 5 + lane; c < p.RF; c += 32)
      o[c] = (obj * p.inv_div) * (dm_sigmoidf(__ldg(q + c)) - (kSparse ? ((c - 5 == sp_class) ? 1.0f : 0.0f) : __ldg(t + c)));
  }
}

// ---- sparse-target mode (SURVEY §8f N3) -------------------------------------------------------------
// GetTargets + GetLoss without the dense y_true: one CTA per image assigns every box (same arithmetic as the dense
// scatter, yolo_targets.cuh), drops the boxes that collide on a record (scatter_nd would sum them and the whole
// record is then zeroed, cds:279-284) and writes the object list the dense path's scan kernel would have found.
__global__ void __launch_bounds__(128) yolo_loss_assign_sparse_kernel(YtParams t, YlParams p, int* __restrict__ keys,
                                                                      float4* __restrict__ sp_t, int32_t* __restrict__ sp_cls,
                                                                      uint32_t* __restrict__ obj_bits) {
  __shared__ int s_cnt[YL_LEVELS];
  const int img = blockIdx.x;
  const int beg = t.offsets[img], end = t.offsets[img + 1];
  if (threadIdx.x < YL_LEVELS) s_cnt[threadIdx.x] = 0;
  for (int i = beg + (int)threadIdx.x; i < end; i += 128) {
    int layer, rin;
    float nx, ny, nw, nh;
    keys[i] = yt_assign(t, i, layer, rin, nx, ny, nw, nh) ? p.lv.anchor_base[layer] + rin : -1;
  }
  __syncthreads();
  // boxes that collide on a record are dropped (all of them): decide for every box first, then retire the keys
  bool dup_mine[8];  // up to 8 * 128 boxes per image in registers; beyond that the flag is recomputed below
  {
    int u = 0;
    for (int i = beg + (int)threadIdx.x; i < end; i += 128, ++u) {
      const int key = keys[i];
      bool dup = false;
      if (key >= 0) for (int j = beg; j < end; ++j) dup |= (j != i) && (keys[j] == key);
      if (u < 8) dup_mine[u] = dup;
    }
  }
  __syncthreads();
  if (end - beg <= 8 * 128) {
    int u = 0;
    for (int i = beg + (int)threadIdx.x; i < end; i += 128, ++u) if (dup_mine[u]) keys[i] = -1;
  } else {
    // rare (more than 1024 boxes in one image): mark duplicates with a sentinel that still compares equal among themselves
    // is not possible in place, so fall back to a serial pass by one thread
    if (threadIdx.x == 0) {
      for (int i = beg; i < end; ++i) {
        const int key = keys[i];
        if (key < 0) continue;
        bool dup = false;
        for (int j = i + 1; j < end; ++j) if (keys[j] == key) { keys[j] = -2; dup = true; }
        if (dup) keys[i] = -2;
      }
    }
  }
  __syncthreads();
  for (int i = beg + (int)threadIdx.x; i < end; i += 128) {
    const int key = keys[i];
    if (key < 0) continue;
    int layer, rin;
    float nx, ny, nw, nh;
    yt_assign(t, i, layer, rin, nx, ny, nw, nh);
    // slot = number of surviving boxes of the same layer with a smaller record index (ascending record order, as the
    // dense path's sorted object list): deterministic run to run, no atomics on the slot
    const int lo_key = p.lv.anchor_base[layer];
    int slot = 0;
    for (int j = beg; j < end; ++j) {
      const int kj = keys[j];
      slot += (kj >= lo_key && kj < key) ? 1 : 0;
    }
    atomicAdd(&s_cnt[layer], 1);
    const size_t gi = (size_t)img * p.n_img + p.lv.anchor_base[layer] + slot;
    p.obj_index[gi] = rin;
    sp_t[gi] = make_float4(nx, ny, nw, nh);
    sp_cls[gi] = t.classes[i];
    atomicOr(obj_bits + (size_t)img * p.bits_words + (key >> 5), 1u << (key & 31));
  }
  __syncthreads();
  if (threadIdx.x < YL_LEVELS) p.gt_count[img * YL_LEVELS + threadIdx.x] = s_cnt[threadIdx.x];
}

// ---- host side ---------------------------------------------------------------------------------
struct YlWs { size_t obj, gt, gtl, cnt, cnt_bytes, part, part_obj, cgrad, oidx, fin, pend, total; int n_cta, n_cta_obj; };

static YlWs yl_layout(const int32_t hw[6], int B, int A, int* n_img_out, YlLevels* lv) {
  YlWs w;
  int n_img = 0, cta = 0, octa = 0;
  for (int l = 0; l < YL_LEVELS; ++l) {
    const int rpi = hw[2 * l] * hw[2 * l + 1] * A;
    const int cpi = (rpi + YL_ICHUNK - 1) / YL_ICHUNK;
    const int ocpi = (rpi + YL_OBJ_CHUNK - 1) / YL_OBJ_CHUNK;
    if (lv) {
      lv->h[l] = hw[2 * l]; lv->w[l] = hw[2 * l + 1]; lv->rec_per_img[l] = rpi; lv->anchor_base[l] = n_img;
      lv->chunks_per_img[l] = cpi; lv->cta_base[l] = cta;
      lv->obj_chunks_per_img[l] = ocpi; lv->obj_cta_base[l] = octa;
    }
    n_img += rpi;
    cta += cpi * B;
    octa += ocpi * B;
  }
  if (lv) { lv->cta_base[YL_LEVELS] = cta; lv->obj_cta_base[YL_LEVELS] = octa; }
  if (n_img_out) *n_img_out = n_img;
  w.n_cta = cta;
  w.n_cta_obj = octa;
  size_t o = 0;
  // zeroed per call: object counts [B,3], the finalize ticket, the pending-record count (+ pad to 8), 3 fixed-point sums
  w.cnt_bytes = b200_align_up(sizeof(int32_t) * ((size_t)B * YL_LEVELS + 2), 8) + 3 * sizeof(unsigned long long) + sizeof(unsigned int) * (size_t)B * YL_LEVELS;
  w.cnt = o; o = b200_align_up(o + w.cnt_bytes, 256);
  w.obj = o; o = b200_align_up(o + sizeof(float) * (size_t)B * n_img, 256);
  w.gt = o; o = b200_align_up(o + sizeof(float4) * (size_t)B * n_img, 256);
  w.gtl = o; o = b200_align_up(o + sizeof(float4) * (size_t)B * n_img, 256);
  w.part = o; o = b200_align_up(o + sizeof(double) * (size_t)cta, 256);
  w.part_obj = o; o = b200_align_up(o + sizeof(double) * 3 * (size_t)YL_LEVELS * B * YL_TERM_SPLIT, 256);
  w.cgrad = o; o = b200_align_up(o + sizeof(float) * (size_t)B * n_img, 256);
  w.oidx = o; o = b200_align_up(o + sizeof(int32_t) * (size_t)B * n_img, 256);
  w.fin = o; o = b200_align_up(o + sizeof(double) * 12 * YL_FIN_CTAS, 256);
  w.pend = o; o = b200_align_up(o + sizeof(uint32_t) * (size_t)B * n_img, 256);
  w.total = o;
  return w;
}

extern "C" size_t b200_yolo_loss_workspace_bytes(const int32_t hw[6], int B, int A) {
  return yl_layout(hw, B, A, nullptr, nullptr).total;
}

struct YlSparseIn {  // ground truth as boxes instead of dense y_true (sparse-target mode)
  const float* boxes; const int32_t* classes; const int32_t* offsets; int total_boxes;
  const float* assign_anchors_wh_host;  // anchors as DataGenerator.GetTargets receives them (may differ in units from the loss's)
};

struct YlSparseWs { size_t sp_t, sp_cls, bits, keys, total; int bits_words; };

static YlSparseWs yl_sparse_layout(size_t dense_total, int B, int n_img, int total_boxes) {
  YlSparseWs w;
  w.bits_words = (n_img + 31) / 32;
  size_t o = b200_align_up(dense_total, 256);
  w.sp_t = o; o = b200_align_up(o + sizeof(float4) * (size_t)B * n_img, 256);
  w.sp_cls = o; o = b200_align_up(o + sizeof(int32_t) * (size_t)B * n_img, 256);
  w.bits = o; o = b200_align_up(o + sizeof(uint32_t) * (size_t)B * w.bits_words, 256);
  w.keys = o; o = b200_align_up(o + sizeof(int32_t) * (size_t)(total_boxes > 0 ? total_boxes : 1), 256);
  w.total = o;
  return w;
}

static int yolo_loss_impl(const float* const y_true[3], const float* const y_pred[3], const int32_t hw[6], int B,
                          int A, int C, const float* anchors_wh_host, const float* image_wh_host,
                          float iou_thresh, int metric, int variant, float batch_divisor, float* out_parts,
                          float* out_loss, unsigned char* out_ignore, float* const out_grad[3], void* workspace,
                          size_t workspace_bytes, void* stream_, const YlSparseIn* sparse = nullptr, int stages = 0xf,
                          const B200Exchange* xchg = nullptr, int publish_only = 0) {
  cudaStream_t stream = (cudaStream_t)stream_;
  B200_REQUIRE((y_true || sparse) && y_pred && hw && anchors_wh_host && image_wh_host && out_loss, B200_ERR_BAD_ARG, "b200_yolo_loss: null argument");
  B200_REQUIRE(B >= 1 && A >= 1 && A <= 8 && C >= 0, B200_ERR_BAD_ARG, "b200_yolo_loss: unsupported shape B=%d A=%d C=%d", B, A, C);
  B200_REQUIRE(metric >= B200_METRIC_YOLO_IOU && metric <= B200_METRIC_YOLO_CIOU, B200_ERR_BAD_ARG,
               "b200_yolo_loss: iou_type must be iou/diou/ciou (metric %d)", metric);
  B200_REQUIRE(variant == YL_VARIANT_TF_YOLO_UTILS || variant == YL_VARIANT_KERAS_YOLO3, B200_ERR_BAD_ARG, "b200_yolo_loss: bad variant %d", variant);
  B200_REQUIRE(batch_divisor > 0.0f, B200_ERR_BAD_ARG, "b200_yolo_loss: batch_divisor must be positive");
  if (out_grad)   // checked before anything is enqueued: a refused call leaves the stream untouched
    for (int l = 0; l < YL_LEVELS; ++l)
      B200_REQUIRE(out_grad[l] && (reinterpret_cast<uintptr_t>(out_grad[l]) & 15) == 0, B200_ERR_BAD_ARG, "%s: grad level %d null or not 16-byte aligned",
                   sparse ? "b200_yolo_loss_from_boxes_grad" : "b200_yolo_loss_grad", l);
  YlParams p;
  int n_img = 0;
  YlWs ws = yl_layout(hw, B, A, &n_img, &p.lv);
  YlSparseWs sws;
  sws.total = ws.total;
  if (sparse) sws = yl_sparse_layout(ws.total, B, n_img, sparse->total_boxes);
  B200_REQUIRE(workspace && workspace_bytes >= sws.total, B200_ERR_WORKSPACE, "b200_yolo_loss: workspace %zu < required %zu", workspace_bytes, sws.total);
  B200_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, B200_ERR_BAD_ARG, "b200_yolo_loss: workspace not 256-byte aligned");
  for (int l = 0; l < YL_LEVELS; ++l) {
    B200_REQUIRE((sparse || y_true[l]) && y_pred[l] && hw[2 * l] > 0 && hw[2 * l + 1] > 0, B200_ERR_BAD_ARG, "b200_yolo_loss: bad level %d", l);
    p.lv.y_true[l] = sparse ? nullptr : y_true[l];
    p.lv.y_pred[l] = y_pred[l];
    for (int a = 0; a < A; ++a) {
      p.lv.anc_w[l][a] = anchors_wh_host[(l * A + a) * 2 + 0];
      p.lv.anc_h[l][a] = anchors_wh_host[(l * A + a) * 2 + 1];
    }
  }
  unsigned char* wsb = static_cast<unsigned char*>(workspace);
  p.B = B; p.A = A; p.C = C; p.RF = 5 + C; p.n_img = n_img;
  // GetLoss scales the width channel by image_wh[::-1] (tyu:48,57, SURVEY Q10): the target log takes tw*image_wh[1] and
  // the predicted width is exp(tw)*anchor_w/image_wh[1].  Yolov4Loss's input_shape[::-1] really is (W, H).  The sparse
  // target assignment (yt_fill_geometry) keeps image_wh in (w, h) order.
  const bool wh_reversed = variant == YL_VARIANT_TF_YOLO_UTILS;
  const float img_w = image_wh_host[wh_reversed ? 1 : 0], img_h = image_wh_host[wh_reversed ? 0 : 1];
  p.img_w = img_w; p.img_h = img_h;
  p.thr = iou_thresh; p.metric = metric; p.variant = variant;
  p.obj_compact = reinterpret_cast<float*>(wsb + ws.obj);
  p.gt_box = reinterpret_cast<float4*>(wsb + ws.gt);
  p.gt_aux = reinterpret_cast<float4*>(wsb + ws.gtl);
  p.log_thr = iou_thresh > 0.0f ? logf(iou_thresh) : 0.0f;
  for (int l = 0; l < YL_LEVELS; ++l)
    for (int a = 0; a < A; ++a)
    {
      p.logk[l][a] = (float)log(((double)p.lv.anc_w[l][a] * (double)p.lv.anc_h[l][a]) / ((double)img_w * (double)img_h));
      // width/height must stay >= 4e-5 (normalised) so that the rounding of x +- w/2 (<= 1.2e-7) is < 0.4 %
      const double tw = log(4e-5 * (double)img_w / (double)p.lv.anc_w[l][a]);
      const double th = log(4e-5 * (double)img_h / (double)p.lv.anc_h[l][a]);
      p.tmin_w[l][a] = (float)(tw > -6.0 ? tw : -6.0);
      p.tmin_h[l][a] = (float)(th > -6.0 ? th : -6.0);
    }
  p.out_ignore = out_ignore;
  p.inv_div = 1.0f / batch_divisor;
  p.conf_grad = out_grad ? reinterpret_cast<float*>(wsb + ws.cgrad) : nullptr;
  p.obj_index = reinterpret_cast<int32_t*>(wsb + ws.oidx);
  p.magic_a = A == 1 ? 0u : (uint32_t)((1ull << 32) / (unsigned long long)A + 1ull);
  for (int l = 0; l < YL_LEVELS; ++l) p.lv.magic_w[l] = p.lv.w[l] == 1 ? 0u : (uint32_t)((1ull << 32) / (unsigned long long)p.lv.w[l] + 1ull);
  p.gt_count = reinterpret_cast<int32_t*>(wsb + ws.cnt);
  p.partials = reinterpret_cast<double*>(wsb + ws.part);
  p.partials_obj = reinterpret_cast<double*>(wsb + ws.part_obj);
  if (stages & 1) B200_CUDA(cudaMemsetAsync(wsb + ws.cnt, 0, ws.cnt_bytes, stream));
  p.pend_queue = reinterpret_cast<uint32_t*>(wsb + ws.pend);
  p.pend_count = reinterpret_cast<unsigned int*>(wsb + ws.cnt) + (size_t)B * YL_LEVELS + 1;
  p.obj_fixed = reinterpret_cast<unsigned long long*>(wsb + ws.cnt + b200_align_up(sizeof(int32_t) * ((size_t)B * YL_LEVELS + 2), 8));
  // full dense call: the scan's last CTA per (image, level) prepares the GT list (stage hooks keep K4a' as its own launch)
  p.scan_ticket = (!sparse && (stages & 3) == 3) ? reinterpret_cast<unsigned int*>(p.obj_fixed + 3) : nullptr;
  p.sp_t = nullptr; p.sp_cls = nullptr; p.obj_bits = nullptr; p.bits_words = 0;
  if (sparse) {
    B200_REQUIRE(sparse->total_boxes >= 0 && sparse->offsets && sparse->assign_anchors_wh_host, B200_ERR_BAD_ARG, "b200_yolo_loss_from_boxes: null box arrays");
    B200_REQUIRE(sparse->total_boxes == 0 || (sparse->boxes && sparse->classes), B200_ERR_BAD_ARG, "b200_yolo_loss_from_boxes: null box arrays");
    B200_REQUIRE((reinterpret_cast<uintptr_t>(sparse->boxes) & 15) == 0, B200_ERR_BAD_ARG, "b200_yolo_loss_from_boxes: boxes not 16-byte aligned");
    YtParams t;
    B200_REQUIRE(yt_fill_geometry(t, A, C, sparse->assign_anchors_wh_host, image_wh_host, hw) == 0, B200_ERR_BAD_ARG, "b200_yolo_loss_from_boxes: bad geometry");
    t.boxes = sparse->boxes; t.classes = sparse->classes; t.offsets = sparse->offsets; t.B = B; t.total = sparse->total_boxes;
    p.bits_words = sws.bits_words;
    float4* sp_t = reinterpret_cast<float4*>(wsb + sws.sp_t);
    int32_t* sp_cls = reinterpret_cast<int32_t*>(wsb + sws.sp_cls);
    uint32_t* bits = reinterpret_cast<uint32_t*>(wsb + sws.bits);
    if (stages & 1) {
      B200_CUDA(cudaMemsetAsync(bits, 0, sizeof(uint32_t) * (size_t)B * sws.bits_words, stream));
      yolo_loss_assign_sparse_kernel<<<B, 128, 0, stream>>>(t, p, reinterpret_cast<int*>(wsb + sws.keys), sp_t, sp_cls, bits);
      B200_LAUNCH_CHECK();
    }
    p.sp_t = sp_t; p.sp_cls = sp_cls; p.obj_bits = bits;
  } else if (stages & 1) {
    yolo_loss_scan_kernel<<<ws.n_cta_obj, YL_CHUNK, 0, stream>>>(p);
    B200_LAUNCH_CHECK();
  }
  if ((stages & 2) && !p.scan_ticket) {
    yolo_loss_gtprep_kernel<<<YL_LEVELS * B, 128, 0, stream>>>(p);
    B200_LAUNCH_CHECK();
  }
  bool use_split = false;
  if (stages & 4) {
    // The split form needs device-resident y_pred, every level 16-byte aligned, and records of >= 8 floats.  Everything
    // else takes the single kernel K4b, which reads pinned host predictions in place over PCIe with one request per record.
    cudaPointerAttributes attr;
    bool host_pred = false;
    if (cudaPointerGetAttributes(&attr, y_pred[YL_LEVELS - 1]) == cudaSuccess) host_pred = attr.type == cudaMemoryTypeHost;
    else (void)cudaGetLastError();
    const int grid = YL_LEVELS * B * YL_TERM_SPLIT + ws.n_cta;
    bool aligned16 = true;
    for (int l = 0; l < YL_LEVELS; ++l) aligned16 &= (reinterpret_cast<uintptr_t>(y_pred[l]) & 15) == 0;
    // Measured at 608x608 batch 64: K4b 71 us; K4b-lean 53.7 us (48 registers, 10 CTAs per SM); the exact pass over the
    // ~12 k undecided records costs 15.6 us as a launch of its own and rides in the widened finalize launch instead.
    use_split = !host_pred && aligned16 && p.RF >= 8;
    if (use_split) {
      // the queue counter and the fixed-point sums are zeroed with the object counts (stage 1); the stage hook may run this
      // pass on its own, repeatedly
      if (!(stages & 1)) B200_CUDA(cudaMemsetAsync(p.pend_count, 0, (size_t)(reinterpret_cast<unsigned char*>(p.obj_fixed + 3) - reinterpret_cast<unsigned char*>(p.pend_count)), stream));
      yolo_loss_ignore_lean_kernel<<<grid, YL_ICHUNK, 0, stream>>>(p);
      if (!(stages & 8)) {   // no finalize in this call: the exact pass as a launch of its own (the finalize launch carries it otherwise)
        B200_LAUNCH_CHECK();
        yolo_loss_ignore_exact_kernel<<<1024, 128, 0, stream>>>(p);
      }
    } else {
      yolo_loss_ignore_kernel<<<grid, YL_ICHUNK, 0, stream>>>(p);
    }
    B200_LAUNCH_CHECK();
  }
  if (!(stages & 8)) return B200_OK;
  YlFinalize f;
  f.partials = p.partials; f.partials_obj = p.partials_obj;
  for (int l = 0; l <= YL_LEVELS; ++l) { f.cta_base[l] = p.lv.cta_base[l]; f.obj_cta_base[l] = l * B * YL_TERM_SPLIT; }
  f.batch_divisor = batch_divisor; f.parts = out_parts; f.loss = out_loss;
  f.slices = reinterpret_cast<double*>(wsb + ws.fin);
  f.ticket = reinterpret_cast<unsigned int*>(wsb + ws.cnt) + (size_t)B * YL_LEVELS;
  f.publish_only = publish_only;
  f.obj_fixed = p.obj_fixed;   // zero unless K4b-exact ran
  if (xchg) f.xchg = *xchg;
  else { f.xchg.rank = 0; f.xchg.world = 1; for (int r = 0; r < B200_XCHG_MAX_WORLD; ++r) f.xchg.mailbox[r] = nullptr; }
  // split form: the finalize launch is widened to 4 CTAs per SM and resolves the queued records first
  int wide = 4 * b200_sm_count();
  if (wide < YL_FIN_CTAS) wide = YL_FIN_CTAS;
  yolo_loss_finalize_kernel<<<use_split ? wide : YL_FIN_CTAS, YL_FIN_THREADS, 0, stream>>>(f, p, use_split ? 1 : 0);
  B200_LAUNCH_CHECK();
  if (out_grad) {
    YlGradDense g;
    g.RF = p.RF;
    unsigned long long cum = 0;
    for (int l = 0; l < YL_LEVELS; ++l) {
      g.records[l] = (unsigned long long)B * p.lv.rec_per_img[l];
      g.grad[l] = out_grad[l];
      g.conf_grad[l] = p.conf_grad + (size_t)B * p.lv.anchor_base[l];
      cum += g.records[l] / 4ull;
      g.quads[l] = cum;
    }
    unsigned long long blocks = (cum + 7) / 8;  // a warp per group of four records
    const unsigned long long cap = (unsigned long long)b200_sm_count() * 64;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    yolo_loss_grad_dense_kernel<<<(int)blocks, 256, 0, stream>>>(g);
    B200_LAUNCH_CHECK();
    if (sparse) yolo_loss_grad_objects_kernel<true><<<B * YL_LEVELS * YL_GRAD_SPLIT, 256, 0, stream>>>(p, out_grad[0], out_grad[1], out_grad[2]);
    else yolo_loss_grad_objects_kernel<false><<<B * YL_LEVELS * YL_GRAD_SPLIT, 256, 0, stream>>>(p, out_grad[0], out_grad[1], out_grad[2]);
    B200_LAUNCH_CHECK();
  }
  return B200_OK;
}

extern "C" int b200_yolo_loss(const float* const y_true[3], const float* const y_pred[3], const int32_t hw[6], int B,
                              int A, int C, const float* anchors_wh_host, const float* image_wh_host,
                              float iou_thresh, int metric, int variant, float batch_divisor, float* out_parts,
                              float* out_loss, unsigned char* out_ignore, void* workspace, size_t workspace_bytes,
                              void* stream_) {
  return yolo_loss_impl(y_true, y_pred, hw, B, A, C, anchors_wh_host, image_wh_host, iou_thresh, metric, variant,
                        batch_divisor, out_parts, out_loss, out_ignore, nullptr, workspace, workspace_bytes, stream_);
}

// Measurement hook: the same call restricted to a subset of its four launches (bit 0 scan, 1 GT prep, 2 ignore + object
// terms, 3 finalize) so that bench.py can time each kernel with CUDA events.  The workspace carries the state between
// the stages; running the stages in order with the same arguments equals one b200_yolo_loss call.
extern "C" int b200_yolo_loss_stages(const float* const y_true[3], const float* const y_pred[3], const int32_t hw[6], int B,
                                     int A, int C, const float* anchors_wh_host, const float* image_wh_host,
                                     float iou_thresh, int metric, int variant, float batch_divisor, float* out_parts,
                                     float* out_loss, void* workspace, size_t workspace_bytes, int stages, void* stream_) {
  B200_REQUIRE(stages > 0 && stages <= 0xf, B200_ERR_BAD_ARG, "b200_yolo_loss_stages: stages must be a non-empty subset of 0xf");
  return yolo_loss_impl(y_true, y_pred, hw, B, A, C, anchors_wh_host, image_wh_host, iou_thresh, metric, variant,
                        batch_divisor, out_parts, out_loss, nullptr, nullptr, workspace, workspace_bytes, stream_, nullptr, stages);
}

extern "C" size_t b200_yolo_loss_from_boxes_workspace_bytes(const int32_t hw[6], int B, int A, int total_boxes) {
  int n_img = 0;
  const YlWs w = yl_layout(hw, B, A, &n_img, nullptr);
  return yl_sparse_layout(w.total, B, n_img, total_boxes).total;
}

extern "C" int b200_yolo_loss_from_boxes(const float* boxes, const int32_t* classes, const int32_t* offsets, int total_boxes,
                                         const float* assign_anchors_wh_host, const float* const y_pred[3], const int32_t hw[6],
                                         int B, int A, int C, const float* anchors_wh_host, const float* image_wh_host,
                                         float iou_thresh, int metric, int variant, float batch_divisor, float* out_parts,
                                         float* out_loss, unsigned char* out_ignore, void* workspace, size_t workspace_bytes,
                                         void* stream_) {
  YlSparseIn sp;
  sp.boxes = boxes; sp.classes = classes; sp.offsets = offsets; sp.total_boxes = total_boxes;
  sp.assign_anchors_wh_host = assign_anchors_wh_host;
  return yolo_loss_impl(nullptr, y_pred, hw, B, A, C, anchors_wh_host, image_wh_host, iou_thresh, metric, variant,
                        batch_divisor, out_parts, out_loss, out_ignore, nullptr, workspace, workspace_bytes, stream_, &sp);
}

// b200_yolo_loss_from_boxes plus d loss / d y_pred, as b200_yolo_loss_grad is to b200_yolo_loss.  The workspace of
// b200_yolo_loss_from_boxes_workspace_bytes already holds the per-record conf gradient the backward reads.
extern "C" int b200_yolo_loss_from_boxes_grad(const float* boxes, const int32_t* classes, const int32_t* offsets, int total_boxes,
                                              const float* assign_anchors_wh_host, const float* const y_pred[3], const int32_t hw[6],
                                              int B, int A, int C, const float* anchors_wh_host, const float* image_wh_host,
                                              float iou_thresh, int metric, int variant, float batch_divisor, float* out_parts,
                                              float* out_loss, float* const out_grad[3], void* workspace, size_t workspace_bytes,
                                              void* stream_) {
  B200_REQUIRE(out_grad, B200_ERR_BAD_ARG, "b200_yolo_loss_from_boxes_grad: null out_grad");
  YlSparseIn sp;
  sp.boxes = boxes; sp.classes = classes; sp.offsets = offsets; sp.total_boxes = total_boxes;
  sp.assign_anchors_wh_host = assign_anchors_wh_host;
  return yolo_loss_impl(nullptr, y_pred, hw, B, A, C, anchors_wh_host, image_wh_host, iou_thresh, metric, variant,
                        batch_divisor, out_parts, out_loss, nullptr, out_grad, workspace, workspace_bytes, stream_, &sp);
}

extern "C" int b200_yolo_loss_grad(const float* const y_true[3], const float* const y_pred[3], const int32_t hw[6],
                                   int B, int A, int C, const float* anchors_wh_host, const float* image_wh_host,
                                   float iou_thresh, int metric, int variant, float batch_divisor, float* out_parts,
                                   float* out_loss, float* const out_grad[3], void* workspace, size_t workspace_bytes,
                                   void* stream_) {
  B200_REQUIRE(out_grad, B200_ERR_BAD_ARG, "b200_yolo_loss_grad: null out_grad");
  return yolo_loss_impl(y_true, y_pred, hw, B, A, C, anchors_wh_host, image_wh_host, iou_thresh, metric, variant,
                        batch_divisor, out_parts, out_loss, nullptr, out_grad, workspace, workspace_bytes, stream_);
}

// Data-parallel forms (SURVEY 8e): every rank passes its own images and batch_divisor = the GLOBAL batch; the 12
// per-level terms are summed over the ranks inside the finalize kernel through the peer mailboxes
// (b200_peer_mailbox_*), so out_parts / out_loss are the global values on every rank and the step has no separate
// collective launch.  y_true == NULL selects the sparse-target form (boxes / classes / offsets as in
// b200_yolo_loss_from_boxes); world == 1 degenerates to the plain calls.
int b200_fill_exchange(B200Exchange& x, int rank, int world, void* const mailboxes[], const char* who);

extern "C" int b200_yolo_loss_dp(const float* const y_true[3], const float* const y_pred[3], const int32_t hw[6], int B,
                                 int A, int C, const float* anchors_wh_host, const float* image_wh_host,
                                 float iou_thresh, int metric, int variant, float global_batch, float* out_parts,
                                 float* out_loss, void* workspace, size_t workspace_bytes, int rank, int world,
                                 void* const mailboxes[], void* stream_) {
  B200Exchange x;
  const int rc = b200_fill_exchange(x, rank, world, mailboxes, "b200_yolo_loss_dp");
  if (rc != B200_OK) return rc;
  return yolo_loss_impl(y_true, y_pred, hw, B, A, C, anchors_wh_host, image_wh_host, iou_thresh, metric, variant,
                        global_batch, out_parts, out_loss, nullptr, nullptr, workspace, workspace_bytes, stream_, nullptr, 0xf, &x);
}

// The same with the exchange split in two: this call ends with the PUBLISH half (out_parts / out_loss hold this rank's
// own terms); b200_yolo_loss_collect_peer, enqueued on any stream ordered behind it, waits for the peers and writes the
// global parts / loss — e.g. on a second stream, under the kernels of the next step.  The publish of step f must be
// ordered after this rank's collect of step f-2 (four slot sets, exchange.cuh).
extern "C" int b200_yolo_loss_dp_publish(const float* const y_true[3], const float* const y_pred[3], const int32_t hw[6], int B,
                                         int A, int C, const float* anchors_wh_host, const float* image_wh_host,
                                         float iou_thresh, int metric, int variant, float global_batch, float* out_parts,
                                         float* out_loss, void* workspace, size_t workspace_bytes, int rank, int world,
                                         void* const mailboxes[], void* stream_) {
  B200Exchange x;
  const int rc = b200_fill_exchange(x, rank, world, mailboxes, "b200_yolo_loss_dp_publish");
  if (rc != B200_OK) return rc;
  return yolo_loss_impl(y_true, y_pred, hw, B, A, C, anchors_wh_host, image_wh_host, iou_thresh, metric, variant,
                        global_batch, out_parts, out_loss, nullptr, nullptr, workspace, workspace_bytes, stream_, nullptr, 0xf, &x, 1);
}

extern "C" int b200_yolo_loss_from_boxes_dp(const float* boxes, const int32_t* classes, const int32_t* offsets, int total_boxes,
                                            const float* assign_anchors_wh_host, const float* const y_pred[3], const int32_t hw[6],
                                            int B, int A, int C, const float* anchors_wh_host, const float* image_wh_host,
                                            float iou_thresh, int metric, int variant, float global_batch, float* out_parts,
                                            float* out_loss, void* workspace, size_t workspace_bytes, int rank, int world,
                                            void* const mailboxes[], void* stream_) {
  B200Exchange x;
  const int rc = b200_fill_exchange(x, rank, world, mailboxes, "b200_yolo_loss_from_boxes_dp");
  if (rc != B200_OK) return rc;
  YlSparseIn sp;
  sp.boxes = boxes; sp.classes = classes; sp.offsets = offsets; sp.total_boxes = total_boxes;
  sp.assign_anchors_wh_host = assign_anchors_wh_host;
  return yolo_loss_impl(nullptr, y_pred, hw, B, A, C, anchors_wh_host, image_wh_host, iou_thresh, metric, variant,
                        global_batch, out_parts, out_loss, nullptr, nullptr, workspace, workspace_bytes, stream_, &sp, 0xf, &x);
}

// loss = sum_l ((xy_l + wh_l) + obj_l) + cls_l from the 12 (all-reduced) terms, in the reference's order of additions
// (tyu:120-125) — the step after b200_allreduce_loss when the NCCL transport is used.
__global__ void yolo_loss_combine_kernel(const float* __restrict__ parts, float* __restrict__ loss) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  float total = 0.0f;
  for (int l = 0; l < 3; ++l)
    total = DM_ADD(total, DM_ADD(DM_ADD(DM_ADD(parts[l * 4 + 0], parts[l * 4 + 1]), parts[l * 4 + 2]), parts[l * 4 + 3]));
  *loss = total;
}

extern "C" int b200_yolo_loss_combine(const float* parts, float* out_loss, void* stream) {
  B200_REQUIRE(parts && out_loss, B200_ERR_BAD_ARG, "b200_yolo_loss_combine: null argument");
  yolo_loss_combine_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(parts, out_loss);
  B200_LAUNCH_CHECK();
  return B200_OK;
}
