// yolo_targets.cuh — best-anchor assignment of one ground-truth box (DataGenerator.GetTargets, datasets/coco_dataset.py:185-245),
// shared by the dense scatter (yolo_targets.cu) and the sparse-target fused loss (yolo_loss.cu).
#pragma once
#include "boxmath.cuh"
#include "common.cuh"

#define YT_LEVELS 3

// GetGroudTruth's corners of a target record (x, y, w, h) (yolo_v4/model.py:380-395): [x - w/2, y - h/2, x + w/2, y + h/2],
// shared by the rows of a dense target (compact.cu) and the rows built from box lists (yolo_loss.cu)
__device__ __forceinline__ void yolo_gt_corners(float x, float y, float w, float h, float* o) {
  const float hw = DM_DIV(w, 2.0f), hh = DM_DIV(h, 2.0f);
  o[0] = DM_SUB(x, hw); o[1] = DM_SUB(y, hh); o[2] = DM_ADD(x, hw); o[3] = DM_ADD(y, hh);
}

struct YtParams {
  const float* boxes;       // [total,4] pixel corners x1,y1,x2,y2
  const int32_t* classes;   // [total]
  const int32_t* offsets;   // [B+1]
  int B, total, A, C, RF, layers_num;
  float img_w, img_h;
  float* target[YT_LEVELS];
  int h[YT_LEVELS], w[YT_LEVELS];
  float anc_w[YT_LEVELS * 8], anc_h[YT_LEVELS * 8];  // flattened (layers*A) in reshape(-1,2) order, pixels
};

// Box i -> (layer, record index within the layer's (H,W,A) grid) and the normalised centre / size stored in the
// record.  Returns false when the cell falls outside the grid (tf.scatter_nd would raise).
__device__ __forceinline__ bool yt_assign(const YtParams& p, int i, int& layer, int& rin, float& nx, float& ny, float& nw, float& nh) {
  const float4 bx = __ldg(reinterpret_cast<const float4*>(p.boxes) + i);
  const float x1 = bx.x, y1 = bx.y, x2 = bx.z, y2 = bx.w;
  // (x2y2 + x1y1) // 2 : float floor division (cds:193)
  const float cx = floorf(DM_DIV(DM_ADD(x2, x1), 2.0f)), cy = floorf(DM_DIV(DM_ADD(y2, y1), 2.0f));
  const float bw = DM_SUB(x2, x1), bh = DM_SUB(y2, y1);
  nx = DM_DIV(cx, p.img_w); ny = DM_DIV(cy, p.img_h);
  nw = DM_DIV(bw, p.img_w); nh = DM_DIV(bh, p.img_h);
  const float mx = DM_DIV(nw, 2.0f), my = DM_DIV(nh, 2.0f);
  const BoxT b = bm_prep(-mx, -my, mx, my, B200_METRIC_YOLO_IOU);
  int best = 0;
  float best_v = 0.f;
  const int n_anchor = YT_LEVELS * p.A;
  for (int k = 0; k < n_anchor; ++k) {
    const float ax = DM_DIV(p.anc_w[k], 2.0f), ay = DM_DIV(p.anc_h[k], 2.0f);
    const BoxT a = bm_prep(-ax, -ay, ax, ay, B200_METRIC_YOLO_IOU);
    const float v = bm_metric(b, a, B200_METRIC_YOLO_IOU);
    if (k == 0 || v > best_v) { best = k; best_v = v; }  // tf.argmax: first maximal index
  }
  layer = best / p.layers_num;
  const int anchor = best % p.layers_num;
  if (layer >= YT_LEVELS || anchor >= p.A) return false;
  const int yy = (int)floorf(DM_MUL(ny, (float)p.h[layer]));
  const int xx = (int)floorf(DM_MUL(nx, (float)p.w[layer]));
  if (yy < 0 || yy >= p.h[layer] || xx < 0 || xx >= p.w[layer]) return false;
  rin = (yy * p.w[layer] + xx) * p.A + anchor;
  return true;
}

// record pointer in the dense targets (nullptr when the box is skipped)
__device__ __forceinline__ float* yt_locate(const YtParams& p, int img, int i, float& nx, float& ny, float& nw, float& nh) {
  int layer, rin;
  if (!yt_assign(p, i, layer, rin, nx, ny, nw, nh)) return nullptr;
  return p.target[layer] + ((size_t)img * p.h[layer] * p.w[layer] * p.A + rin) * p.RF;
}

// host: fills the geometry part of YtParams (targets may be null pointers for the sparse path)
static inline int yt_fill_geometry(YtParams& p, int A, int C, const float* anchors_wh_host, const float* image_wh_host, const int32_t hw[6]) {
  if (A < 1 || A > 8 || C < 0 || !anchors_wh_host || !image_wh_host || !hw) return -1;
  p.A = A; p.C = C; p.RF = 5 + C;
  p.layers_num = YT_LEVELS;  // tf.shape(anchors_wh)[0], cds:191
  p.img_w = image_wh_host[0]; p.img_h = image_wh_host[1];
  for (int l = 0; l < YT_LEVELS; ++l) {
    if (hw[2 * l] <= 0 || hw[2 * l + 1] <= 0) return -1;
    p.target[l] = nullptr; p.h[l] = hw[2 * l]; p.w[l] = hw[2 * l + 1];
  }
  for (int k = 0; k < YT_LEVELS * A; ++k) { p.anc_w[k] = anchors_wh_host[2 * k]; p.anc_h[k] = anchors_wh_host[2 * k + 1]; }
  return 0;
}
