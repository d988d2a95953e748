// effdet_anchor.cuh — the EfficientDet anchor of a (level, y, x, a) rebuilt from the per-level table, and the
// _boxes_encoder of one (anchor, GT box) pair.  Shared by the target assignment (effdet.cu) and the loss computed
// straight from box lists (effdet_loss.cu), so that both produce the same anchors and the same box targets.
//
// Anchors are never read from HBM: every kernel rebuilds an anchor box from a tiny per-level table
// (row centres yc[H], column centres xc[W], half extents hy[A], hx[A]; built on the host with the reference's own
// double-precision Python arithmetic) exactly as the reference does — box = [yc-hy, xc-hx, yc+hy, xc+hx] in fp32,
// then centre/size re-derived from those corners (anc:204-217) — so results are bit-identical to reading
// Anchors.boxes while saving 0.8 MB (D0) / 7 MB (D7) of reads per image.
#pragma once
#include "common.cuh"
#include "detmath.h"

#define EF_MAX_LEVELS 8

struct EfLevels {
  int num_levels, A;
  int h[EF_MAX_LEVELS], w[EF_MAX_LEVELS];
  int anc_per_img[EF_MAX_LEVELS];   // h*w*A
  int anchor_base[EF_MAX_LEVELS];   // flat anchor index of the level's first anchor within an image
  const float* table;               // device
  int tab_off[EF_MAX_LEVELS];       // float offset of the level's [yc(h) | xc(w) | hy(A) | hx(A)] block
};

struct AnchorBox { float y1, x1, y2, x2; };

__device__ __forceinline__ AnchorBox ef_anchor(const EfLevels& lv, int l, int y, int x, int a) {
  const float* t = lv.table + lv.tab_off[l];
  const float yc = __ldg(t + y), xc = __ldg(t + lv.h[l] + x);
  const float hy = __ldg(t + lv.h[l] + lv.w[l] + a), hx = __ldg(t + lv.h[l] + lv.w[l] + lv.A + a);
  AnchorBox b;
  b.y1 = DM_SUB(yc, hy); b.x1 = DM_SUB(xc, hx); b.y2 = DM_ADD(yc, hy); b.x2 = DM_ADD(xc, hx);  // anc:77-78
  return b;
}

__device__ __forceinline__ void ef_split(const EfLevels& lv, int l, int rin, int& y, int& x, int& a) {
  const int cell = rin / lv.A;
  a = rin - cell * lv.A;
  y = cell / lv.w[l];
  x = cell - y * lv.w[l];
}

// _boxes_encoder (anc:231-243): the box target (ty, tx, th, tw) of anchor (ay1, ax1, ay2, ax2) for GT (by1, bx1, by2, bx2)
__device__ __forceinline__ float4 ef_encode_box(float ay1, float ax1, float ay2, float ax2, float by1, float bx1, float by2,
                                                float bx2) {
  const float yca = DM_DIV(DM_ADD(ay2, ay1), 2.0f), xca = DM_DIV(DM_ADD(ax2, ax1), 2.0f);
  const float ha = dm_max(1e-8f, DM_SUB(ay2, ay1)), wa = dm_max(1e-8f, DM_SUB(ax2, ax1));
  const float yc = DM_DIV(DM_ADD(by2, by1), 2.0f), xc = DM_DIV(DM_ADD(bx2, bx1), 2.0f);
  const float h = dm_max(1e-8f, DM_SUB(by2, by1)), w = dm_max(1e-8f, DM_SUB(bx2, bx1));
  return make_float4(DM_DIV(DM_SUB(yc, yca), ha), DM_DIV(DM_SUB(xc, xca), wa), dm_logf(DM_DIV(h, ha)), dm_logf(DM_DIV(w, wa)));
}

// Host: the level description of hw = {H0,W0,H1,W1,...}; returns the anchors per image, or -1 for a bad spec.
static inline int ef_fill_levels(EfLevels& lv, int num_levels, const int32_t* hw, int A, const float* table_dev) {
  if (num_levels < 1 || num_levels > EF_MAX_LEVELS || A < 1) return -1;
  lv.num_levels = num_levels; lv.A = A; lv.table = table_dev;
  int base = 0, off = 0;
  for (int l = 0; l < EF_MAX_LEVELS; ++l) {
    if (l < num_levels) {
      lv.h[l] = hw[2 * l]; lv.w[l] = hw[2 * l + 1];
      if (lv.h[l] <= 0 || lv.w[l] <= 0) return -1;
      lv.anc_per_img[l] = lv.h[l] * lv.w[l] * A;
      lv.anchor_base[l] = base; base += lv.anc_per_img[l];
      lv.tab_off[l] = off; off += lv.h[l] + lv.w[l] + 2 * A;
    } else {
      lv.h[l] = lv.w[l] = 1; lv.anc_per_img[l] = 0; lv.anchor_base[l] = base; lv.tab_off[l] = off;
    }
  }
  return base;
}
