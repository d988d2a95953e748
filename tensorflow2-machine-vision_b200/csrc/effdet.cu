// effdet.cu — EfficientDet head utilities: anchors, box decode, per-image post-processing, target assignment.
//
// Replaces (paths relative to AIServer/ai_api/ai_models/):
//   efficientnet/utils/anchors.py:46-84    Anchors._generate_boxes        -> effdet_anchors_kernel
//   efficientnet/utils/anchors.py:141-158, 245-274  convert_outputs_boxes / _boxes_decoder -> effdet_decode_kernel
//   efficientnet/utils/anchors.py:161-202  convert_outputs_one            -> effdet_filter_kernel + effdet_nms_finalize_kernel
//   efficientnet/utils/anchors.py:91-138, 219-243   generate_targets / _boxes_encoder -> effdet_assign_kernel
//
// The filter streams its class logits through the per-warp WarpSlabRing of bulkcopy.cuh, the same ring as the YOLO filter;
// the filter and the fused eval-step stream share one box decode (ef_decode_box) and append to the candidate store of
// nms.cuh (CandStore: workspace layout, append and NMS output tail, shared with yolo_decode.cu; EfficientDet adds the
// buffers of the multi-CTA pre-selection).
//
// Anchors are rebuilt in-kernel from the per-level table (effdet_anchor.cuh, shared with effdet_loss.cu).
#include "nms.cuh"
#include "effdet_focal.cuh"
#include "effdet_anchor.cuh"
#include "bulkcopy.cuh"

#define EF_STAGES 2

// _boxes_decoder (anc:245-274): the box of anchor `an` from its head offsets rel = (ty, tx, th, tw)
__device__ __forceinline__ float4 ef_decode_box(const AnchorBox& an, float4 rel) {
  const float yca = DM_DIV(DM_ADD(an.y2, an.y1), 2.0f), xca = DM_DIV(DM_ADD(an.x2, an.x1), 2.0f);
  const float ha = DM_SUB(an.y2, an.y1), wa = DM_SUB(an.x2, an.x1);
  const float w = DM_MUL(dm_expf(rel.w), wa), h = DM_MUL(dm_expf(rel.z), ha);
  const float yc = DM_ADD(DM_MUL(rel.x, ha), yca), xc = DM_ADD(DM_MUL(rel.y, wa), xca);
  const float hh = DM_DIV(h, 2.0f), hw = DM_DIV(w, 2.0f);
  return make_float4(DM_SUB(yc, hh), DM_SUB(xc, hw), DM_ADD(yc, hh), DM_ADD(xc, hw));
}

// ---- anchors -------------------------------------------------------------------------------------
__global__ void effdet_anchors_kernel(EfLevels lv, int l, float4* __restrict__ out) {
  const int n = lv.anc_per_img[l];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int y, x, a;
    ef_split(lv, l, i, y, x, a);
    const AnchorBox b = ef_anchor(lv, l, y, x, a);
    out[i] = make_float4(b.y1, b.x1, b.y2, b.x2);
  }
}

// ---- decode (anc:245-274) ---------------------------------------------------------------------------
struct EfDecodeParams {
  EfLevels lv;
  int B;
  const float4* rel[EF_MAX_LEVELS];
  float4* out[EF_MAX_LEVELS];
  long long elem_base[EF_MAX_LEVELS + 1];  // cumulative B*anc_per_img
};

__global__ void __launch_bounds__(256) effdet_decode_kernel(EfDecodeParams p) {
  const long long total = p.elem_base[p.lv.num_levels];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int l = 0;
#pragma unroll
    for (int k = 1; k < EF_MAX_LEVELS; ++k) if (k < p.lv.num_levels && i >= p.elem_base[k]) l = k;
    const long long e = i - p.elem_base[l];
    const unsigned int api = (unsigned int)p.lv.anc_per_img[l];
    const unsigned int img = (unsigned int)(e / api);  // e < 2^31*api in practice; 64/32 division only here
    const int rin = (int)(e - (long long)img * api);
    int y, x, a;
    ef_split(p.lv, l, rin, y, x, a);
    const AnchorBox an = ef_anchor(p.lv, l, y, x, a);
    const float4 r = __ldcs(p.rel[l] + e);
    const float4 b = ef_decode_box(an, r);
    __stcs(p.out[l] + e, b);
  }
}

// ---- class argmax / background filter (anc:168-189), streaming like yolo_decode_filter_kernel ----------
struct EfFilterParams {
  EfLevels lv;
  int B0, NB, C;                 // images [B0, B0+NB) of a batch of size B
  int B;
  const float* cls[EF_MAX_LEVELS];    // (B,H,W,A,C) logits
  const float4* boxes[EF_MAX_LEVELS]; // (B,H,W,A,4) decoded, or null: decode here from rel (lv.table must be set)
  const float4* rel[EF_MAX_LEVELS];   // (B,H,W,A,4) head offsets ty,tx,th,tw (fused decode mode)
  float4* dec[EF_MAX_LEVELS];         // fused decode mode: the dense decoded tensor is written here (may be null)
  long long tile_base[EF_MAX_LEVELS + 1];  // tiles of 32 anchors over the NB images of each level
  CandStore st;                  // [NB] images
};

__global__ void __launch_bounds__(256, 1) effdet_filter_kernel(EfFilterParams p) {
  extern __shared__ __align__(128) unsigned char ef_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
  const int C = p.C;
  WarpSlabRing<EF_STAGES> ring(ef_smem, C);
  const long long n_tiles = p.tile_base[p.lv.num_levels];
  const long long gwarp = (long long)blockIdx.x * wpc + warp, gstride = (long long)gridDim.x * wpc;

  auto locate = [&](long long tile, int& l, long long& rec0, int& nrec) {
    l = 0;
#pragma unroll
    for (int k = 1; k < EF_MAX_LEVELS; ++k) if (k < p.lv.num_levels && tile >= p.tile_base[k]) l = k;
    rec0 = (tile - p.tile_base[l]) * 32;  // record index within the NB-image slice of level l
    const long long remain = (long long)p.NB * p.lv.anc_per_img[l] - rec0;
    nrec = remain < 32 ? (int)remain : 32;
  };
  auto issue = [&](long long tile, int s) {
    int l, nrec; long long rec0;
    locate(tile, l, rec0, nrec);
    ring.issue(s, p.cls[l] + ((long long)p.B0 * p.lv.anc_per_img[l] + rec0) * C, nrec, C);
  };
  long long t_issue = gwarp;
#pragma unroll
  for (int s = 0; s < EF_STAGES; ++s) { if (t_issue < n_tiles) issue(t_issue, s); t_issue += gstride; }
  for (long long tile = gwarp; tile < n_tiles; tile += gstride) {
    ring.wait();
    int l, nrec; long long rec0;
    locate(tile, l, rec0, nrec);
    const float* r = ring.slab(ring.stage) + lane * C;
    bool pass = false;
    int img = 0, cls = 0;
    float score = 0.f;
    uint32_t aidx = 0;
    float4 box = make_float4(0.f, 0.f, 0.f, 0.f);
    const bool fused_decode = p.rel[l] != nullptr;   // block-uniform
    int rin = 0, mi = 0;
    long long grec = 0;
    float m = 0.f;
    float4 r4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (lane < nrec) {
      const long long rec = rec0 + lane;
      const int api = p.lv.anc_per_img[l];
      const long long total = (long long)p.NB * api;
      if (total < 0x7fffffffLL) { img = (int)((uint32_t)rec / (uint32_t)api); rin = (int)((uint32_t)rec - (uint32_t)img * (uint32_t)api); }
      else { img = (int)(rec / api); rin = (int)(rec - (long long)img * api); }
      grec = (long long)(p.B0 + img) * api + rin;
      if (fused_decode) r4 = __ldcs(p.rel[l] + grec);   // issued before the class scan: coalesced, 16 bytes per lane
      // tf.math.argmax: first maximal index; reduce_max: the maximum (anc:172-174)
      m = r[0];
      for (int c = 1; c < C; ++c) { const float v = r[c]; if (v > m) { m = v; mi = c; } }
    }
    // the class scan was the last read of the slab: its refill is in flight during the decode and the append below
    __syncwarp();
    if (t_issue < n_tiles) issue(t_issue, ring.stage);
    t_issue += gstride;
    if (lane < nrec) {
      if (fused_decode) {
        // convert_outputs_boxes for every anchor: the dense decoded tensor is an output
        int y, x, an_i;
        ef_split(p.lv, l, rin, y, x, an_i);
        box = ef_decode_box(ef_anchor(p.lv, l, y, x, an_i), r4);
        if (p.dec[l]) __stcs(p.dec[l] + grec, box);
      }
      if (mi != 0) {  // classes_mask = classes_id != 0 (anc:179)
        pass = true; cls = mi; score = m;
        aidx = (uint32_t)(p.lv.anchor_base[l] + rin);
        if (!fused_decode) box = __ldg(p.boxes[l] + grec);
      }
    }
    warp_append_by_image(p.st, pass, img, aidx, [&](size_t slot) {
      p.st.box[slot] = box; p.st.score[slot] = score; p.st.cls[slot] = cls;
    });
    ring.advance();
  }
}

struct EfFinalizeParams {
  NmsConfig cfg;
  CandStore st;
  float* out_boxes; long long* out_cls; float* out_score; int32_t* out_sel_idx; int32_t* out_sel_anchor; int32_t* out_count;
};

template <int METRIC>
__global__ void __launch_bounds__(NMS_THREADS, 1) effdet_nms_finalize_kernel(EfFinalizeParams p) {
  extern __shared__ __align__(16) unsigned char nms_smem[];
  const int img = blockIdx.x;
  const size_t cbase = (size_t)img * p.st.n_img;
  int32_t* pos = p.st.pos + (size_t)img * p.cfg.max_out;
  NmsPre pre;
  if (p.st.pre_keys) {
    pre.keys = p.st.pre_keys + (size_t)img * NMS_PRE_CAP; pre.pos = p.st.pre_pos + (size_t)img * NMS_PRE_CAP;
    pre.count = p.st.pre_count + img; pre.eligible = p.st.pre_elig + img; pre.khi = p.st.pre_khi + img;
  }
  const int kept = nms_run_segment<METRIC, NmsLoadDirectAgnostic>(cand_segment(p.st, img, false), p.cfg, pos, nms_smem,
                                                                  p.st.pre_keys ? &pre : nullptr);
  __syncthreads();
  if (threadIdx.x == 0) p.out_count[img] = kept;
  const size_t obase = (size_t)img * p.cfg.max_out;
  uint32_t* wprefix = reinterpret_cast<uint32_t*>(nms_smem);
  cand_word_prefix(p.st, img, wprefix);
  for (int k = threadIdx.x; k < kept; k += blockDim.x) {
    const int q = pos[k];
    reinterpret_cast<float4*>(p.out_boxes)[obase + k] = p.st.box[cbase + q];
    p.out_cls[obase + k] = (long long)p.st.cls[cbase + q];               // tf.argmax -> int64 (anc:172)
    p.out_score[obase + k] = dm_sigmoidf(p.st.score[cbase + q]);          // sigmoid only on survivors (anc:200)
    const uint32_t a = p.st.aidx[cbase + q];
    if (p.out_sel_anchor) p.out_sel_anchor[obase + k] = (int32_t)a;
    if (p.out_sel_idx) p.out_sel_idx[obase + k] = cand_sel_idx(p.st, img, wprefix, a);
  }
}

// ---- target assignment (anc:91-138) ------------------------------------------------------------------
struct EfAssignParams {
  EfLevels lv;
  int B, C;
  uint32_t magic_c;           // floor(2^32/C)+1 (exact quotient for dividends below 2^16 * C)
  float thr;
  const float* gt_boxes;      // [total,4] yxyx
  const int32_t* gt_classes;  // [total]
  const int32_t* gt_offsets;  // [B+1]
  float4* out_boxes[EF_MAX_LEVELS];        // (B,H,W,A,4)
  float* out_onehot[EF_MAX_LEVELS];        // (B,H,W,A,C), or null when out_class is used
  int32_t* out_class[EF_MAX_LEVELS];       // (B,H,W,A): class id instead of the one-hot row (sparse-target mode)
  unsigned char* out_mask[EF_MAX_LEVELS];  // (B,H,W,A,1)
  int32_t* out_match;                      // match mode: the matched row of gt_boxes (or -1) per anchor, level l at B*anchor_base[l]
  double* positives;                       // match mode: += matched anchors
  int cta_base[EF_MAX_LEVELS + 1];         // CTAs of 256 anchors, per (level, image)
  int chunks_per_img[EF_MAX_LEVELS];
};

#define EF_GT_TILE 128

__global__ void __launch_bounds__(256, 8) effdet_assign_kernel(EfAssignParams p) {
  __shared__ float4 s_gt[EF_GT_TILE];
  __shared__ float s_ga[EF_GT_TILE];
  int l = 0;
#pragma unroll
  for (int k = 1; k < EF_MAX_LEVELS; ++k) if (k < p.lv.num_levels && (int)blockIdx.x >= p.cta_base[k]) l = k;
  const int rc = blockIdx.x - p.cta_base[l];
  const int img = rc / p.chunks_per_img[l];
  const int chunk = rc - img * p.chunks_per_img[l];
  const int api = p.lv.anc_per_img[l];
  const int rin = chunk * 256 + (int)threadIdx.x;
  const bool active = rin < api;
  const int g_beg = p.gt_offsets[img], n_gt = p.gt_offsets[img + 1] - g_beg;
  BoxT an;
  an.c0 = an.c1 = an.c2 = an.c3 = an.area = an.at = 0.f;
  if (active) {
    int y, x, a;
    ef_split(p.lv, l, rin, y, x, a);
    const AnchorBox b = ef_anchor(p.lv, l, y, x, a);
    an = bm_prep(b.y1, b.x1, b.y2, b.x2, B200_METRIC_EFF_IOU);
  }
  // Bounding box of the CTA's 256 anchors (a run of cells of one row): a GT that does not overlap it has IoU exactly 0
  // with every anchor here and, for thr > 0, can neither match nor change the outcome (an all-zero row stays
  // unmatched whatever its argmax), so each GT tile is culled once per CTA and the anchors walk only the survivors —
  // in ascending GT order, which keeps tf.argmax's first-maximal-index rule.
  __shared__ float s_bb[8][4];
  __shared__ uint32_t s_mask[EF_GT_TILE / 32];
  {
    float y1 = active ? an.c0 : INFINITY, x1 = active ? an.c1 : INFINITY;
    float y2 = active ? an.c2 : -INFINITY, x2 = active ? an.c3 : -INFINITY;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      y1 = fminf(y1, __shfl_xor_sync(0xffffffffu, y1, o)); x1 = fminf(x1, __shfl_xor_sync(0xffffffffu, x1, o));
      y2 = fmaxf(y2, __shfl_xor_sync(0xffffffffu, y2, o)); x2 = fmaxf(x2, __shfl_xor_sync(0xffffffffu, x2, o));
    }
    if ((threadIdx.x & 31) == 0) { float* d = s_bb[threadIdx.x >> 5]; d[0] = y1; d[1] = x1; d[2] = y2; d[3] = x2; }
  }
  __syncthreads();
  float by1 = s_bb[0][0], bx1 = s_bb[0][1], by2 = s_bb[0][2], bx2 = s_bb[0][3];
#pragma unroll
  for (int w = 1; w < 8; ++w) {
    by1 = fminf(by1, s_bb[w][0]); bx1 = fminf(bx1, s_bb[w][1]); by2 = fmaxf(by2, s_bb[w][2]); bx2 = fmaxf(bx2, s_bb[w][3]);
  }
  const bool cull = p.thr > 0.0f;
  float best = -INFINITY;
  int best_i = 0;
  for (int g0 = 0; g0 < n_gt; g0 += EF_GT_TILE) {
    const int m = min(EF_GT_TILE, n_gt - g0);
    __syncthreads();
    if (threadIdx.x < EF_GT_TILE) {
      bool relevant = false;
      if ((int)threadIdx.x < m) {
        const float* q = p.gt_boxes + 4 * (size_t)(g_beg + g0 + threadIdx.x);
        const BoxT g = bm_prep(q[0], q[1], q[2], q[3], B200_METRIC_EFF_IOU);
        s_gt[threadIdx.x] = make_float4(g.c0, g.c1, g.c2, g.c3);
        s_ga[threadIdx.x] = g.area;
        // positive overlap with the bounding box in both axes (false for NaN coordinates, which can never be chosen)
        relevant = !cull || ((DM_SUB(dm_min(by2, g.c2), dm_max(by1, g.c0)) > 0.0f) && (DM_SUB(dm_min(bx2, g.c3), dm_max(bx1, g.c1)) > 0.0f));
      }
      const uint32_t bits = __ballot_sync(0xffffffffu, relevant);
      if ((threadIdx.x & 31) == 0) s_mask[threadIdx.x >> 5] = bits;
    }
    __syncthreads();
    if (active) {
#pragma unroll
      for (int w = 0; w < EF_GT_TILE / 32; ++w) {
        uint32_t bits = s_mask[w];
        while (bits) {
          const int g = (w << 5) + __ffs(bits) - 1;
          bits &= bits - 1u;
          const float4 c = s_gt[g];
          // clamped intersection extents (eiou:58-64); zero overlap -> iou = divide_no_nan(0, union) = +0 exactly
          const float iw = dm_max(0.0f, DM_SUB(dm_min(an.c3, c.w), dm_max(an.c1, c.y)));
          const float ih = dm_max(0.0f, DM_SUB(dm_min(an.c2, c.z), dm_max(an.c0, c.x)));
          float v = 0.0f;
          if (iw > 0.0f && ih > 0.0f) {
            const float inter = DM_MUL(iw, ih);
            v = bm_dnn(inter, DM_SUB(DM_ADD(an.area, s_ga[g]), inter));
          } else if (!(iw == iw) || !(ih == ih)) {
            BoxT gb; gb.c0 = c.x; gb.c1 = c.y; gb.c2 = c.z; gb.c3 = c.w; gb.area = s_ga[g]; gb.at = 0.f;
            v = bm_metric(an, gb, B200_METRIC_EFF_IOU);
          }
          if (v > best) { best = v; best_i = g0 + g; }  // tf.argmax: first maximal index
        }
      }
    }
  }
  // encode + outputs
  const bool matched = active && (n_gt > 0) && (best >= p.thr);  // iou_max >= thr (anc:121)
  const size_t abase = (size_t)img * api;
  if (p.out_match) {  // match mode (block-uniform): the GT row stands for the targets, the loss pass encodes them itself
    if (active) p.out_match[(size_t)p.B * p.lv.anchor_base[l] + abase + rin] = matched ? g_beg + best_i : -1;
    const int n = __syncthreads_count(matched);
    if (threadIdx.x == 0 && n > 0) atomicAdd(p.positives, (double)n);  // integer-valued: exact and order-independent
    return;
  }
  int cls = 0;
  float4 enc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (matched) {
    const float* q = p.gt_boxes + 4 * (size_t)(g_beg + best_i);
    cls = p.gt_classes[g_beg + best_i];
    enc = ef_encode_box(an.c0, an.c1, an.c2, an.c3, q[0], q[1], q[2], q[3]);
  }
  if (active) {
    p.out_boxes[l][abase + rin] = enc;
    p.out_mask[l][abase + rin] = matched ? 1 : 0;
  }
  if (p.out_class[l]) {  // sparse-target mode: the class id stands for the one-hot row (block-uniform branch)
    if (active) p.out_class[l][abase + rin] = cls;
    return;
  }
  // one-hot rows (C floats per anchor, class 0 = background for unmatched anchors, anc:131-133; tf.one_hot: out of
  // range -> zeros): the CTA's 256 rows are one contiguous span of rows*C floats, written once with aligned 16-byte
  // streaming stores; the 1.0 of row r sits at flat element r*C + cls[r] of the span.
  __shared__ int s_hot[256];
  s_hot[threadIdx.x] = (active && cls >= 0 && cls < p.C) ? (int)threadIdx.x * p.C + cls : -1;
  __syncthreads();
  const int rows = min(256, api - chunk * 256);
  float* dst = p.out_onehot[l] + (abase + (size_t)chunk * 256) * p.C;
  const int n_el = rows * p.C;
  const int head = min(n_el, (int)(((16u - ((unsigned)(uintptr_t)dst & 15u)) & 15u) >> 2));
  const int n_vec = p.C >= 3 ? (n_el - head) >> 2 : 0;  // rows narrower than 3 take the scalar path below
  float4* dst4 = reinterpret_cast<float4*>(dst + head);
  for (int i = threadIdx.x; i < n_vec; i += 256) {
    const int e = head + 4 * i;                                   // first flat element of this float4
    const int r = (int)__umulhi((uint32_t)e, p.magic_c);          // e / C (magic_c = floor(2^32/C)+1, e < 2^16 * C)
    const int h0 = s_hot[r], h1 = (r + 1 < rows) ? s_hot[r + 1] : -1;  // a float4 touches at most rows r and r+1 when C >= 3
    float4 v;
    v.x = (e == h0 || e == h1) ? 1.0f : 0.0f;
    v.y = (e + 1 == h0 || e + 1 == h1) ? 1.0f : 0.0f;
    v.z = (e + 2 == h0 || e + 2 == h1) ? 1.0f : 0.0f;
    v.w = (e + 3 == h0 || e + 3 == h1) ? 1.0f : 0.0f;
    __stcs(dst4 + i, v);
  }
  // unaligned head / tail elements (and every element of rows narrower than 3): scalar stores
  for (int e = threadIdx.x; e < n_el; e += 256) {
    if (e >= head && e < head + (n_vec << 2)) continue;
    const int r = e / p.C;
    dst[e] = (s_hot[r] == e) ? 1.0f : 0.0f;
  }
}

// ---- host side ------------------------------------------------------------------------------------
extern "C" size_t b200_effdet_table_floats(int num_levels, const int32_t* hw, int A) {
  size_t n = 0;
  for (int l = 0; l < num_levels; ++l) n += (size_t)hw[2 * l] + hw[2 * l + 1] + 2 * (size_t)A;
  return n;
}

extern "C" int b200_effdet_anchors(int num_levels, const int32_t* hw, int A, const float* table_dev, int level,
                                   float* out, void* stream) {
  EfLevels lv;
  B200_REQUIRE(hw && table_dev && out, B200_ERR_BAD_ARG, "b200_effdet_anchors: null argument");
  B200_REQUIRE(ef_fill_levels(lv, num_levels, hw, A, table_dev) >= 0, B200_ERR_BAD_ARG, "b200_effdet_anchors: bad level spec");
  B200_REQUIRE(level >= 0 && level < num_levels, B200_ERR_BAD_ARG, "b200_effdet_anchors: bad level %d", level);
  B200_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, B200_ERR_BAD_ARG, "b200_effdet_anchors: out not 16-byte aligned");
  const int n = lv.anc_per_img[level];
  effdet_anchors_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(lv, level, reinterpret_cast<float4*>(out));
  B200_LAUNCH_CHECK();
  return B200_OK;
}

extern "C" int b200_effdet_decode(int num_levels, const int32_t* hw, int A, const float* table_dev, int B,
                                  const float* const rel[], float* const out[], void* stream) {
  EfDecodeParams p;
  B200_REQUIRE(hw && table_dev && rel && out, B200_ERR_BAD_ARG, "b200_effdet_decode: null argument");
  B200_REQUIRE(ef_fill_levels(p.lv, num_levels, hw, A, table_dev) >= 0, B200_ERR_BAD_ARG, "b200_effdet_decode: bad level spec");
  B200_REQUIRE(B >= 0, B200_ERR_BAD_ARG, "b200_effdet_decode: negative batch");
  if (B == 0) return B200_OK;
  p.B = B;
  long long cum = 0;
  for (int l = 0; l < EF_MAX_LEVELS; ++l) {
    p.elem_base[l] = cum;
    if (l < num_levels) {
      B200_REQUIRE(rel[l] && out[l], B200_ERR_BAD_ARG, "b200_effdet_decode: null level %d", l);
      B200_REQUIRE(((reinterpret_cast<uintptr_t>(rel[l]) | reinterpret_cast<uintptr_t>(out[l])) & 15) == 0, B200_ERR_BAD_ARG,
                   "b200_effdet_decode: level %d not 16-byte aligned", l);
      p.rel[l] = reinterpret_cast<const float4*>(rel[l]);
      p.out[l] = reinterpret_cast<float4*>(out[l]);
      cum += (long long)B * p.lv.anc_per_img[l];
    } else { p.rel[l] = nullptr; p.out[l] = nullptr; }
  }
  p.elem_base[EF_MAX_LEVELS] = cum;
  for (int l = num_levels; l <= EF_MAX_LEVELS; ++l) p.elem_base[l] = cum;
  long long blocks = (cum + 255) / 256;
  const long long cap = (long long)b200_sm_count() * 64;  // many short CTAs: see el_cta_plan
  if (blocks > cap) blocks = cap;
  effdet_decode_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(p);
  B200_LAUNCH_CHECK();
  return B200_OK;
}

__global__ void __launch_bounds__(NMS_THREADS, 1) effdet_nms_pivot_kernel(NmsPreselectParams p) {
  extern __shared__ __align__(16) unsigned char pre_smem[];
  nms_pivot_body(p, pre_smem);
}
__global__ void __launch_bounds__(256) effdet_nms_pregather_kernel(NmsPreselectParams p) { nms_pregather_body(p); }

// The NMS tail shared by b200_effdet_postprocess and the fused entry points: (large segments) pivot + multi-CTA
// pre-gather of the first window, then one CTA per image.
static int ef_launch_nms(const CandStore& st, int num_images, int max_out, float iou_thr, float score_thr, int metric,
                         float* out_boxes, long long* out_class_id, float* out_score, int32_t* out_sel_idx,
                         int32_t* out_sel_anchor, int32_t* out_count, cudaStream_t stream) {
  EfFinalizeParams np;
  np.cfg.metric = metric; np.cfg.mode = B200_NMS_AGNOSTIC; np.cfg.iou_thr = iou_thr; np.cfg.score_thr = score_thr;
  np.cfg.use_score_thr = 1; np.cfg.max_out = max_out;
  np.st = st;
  if (st.pre_keys) {
    // large segments: several CTAs per image gather the first NMS window so the single NMS CTA does not have to
    // scan hundreds of thousands of scores alone
    NmsPreselectParams pp;
    int slices = (5 * b200_sm_count() + num_images - 1) / num_images;   // ~5 CTAs of 256 threads (46 registers) per SM: one wave
    if (slices < 1) slices = 1;
    if (slices > 64) slices = 64;
    pp.scores = st.score; pp.order_id = st.aidx; pp.counts = st.counts; pp.stride = st.n_img; pp.slices = slices;
    pp.use_score_thr = 1; pp.score_thr = score_thr;
    pp.keys = st.pre_keys; pp.pos = st.pre_pos; pp.count = st.pre_count; pp.eligible = st.pre_elig; pp.khi = st.pre_khi;
    B200_CUDA(cudaFuncSetAttribute(effdet_nms_pivot_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)NMS_PIVOT_SMEM));
    effdet_nms_pivot_kernel<<<num_images, NMS_THREADS, NMS_PIVOT_SMEM, stream>>>(pp);
    B200_LAUNCH_CHECK();
    effdet_nms_pregather_kernel<<<num_images * slices, 256, 0, stream>>>(pp);
    B200_LAUNCH_CHECK();
  }
  np.out_boxes = out_boxes; np.out_cls = out_class_id; np.out_score = out_score; np.out_sel_idx = out_sel_idx;
  np.out_sel_anchor = out_sel_anchor; np.out_count = out_count;
  const size_t smem2 = cand_finalize_smem_bytes(st, max_out);
  B200_REQUIRE(smem2 <= 220 * 1024, B200_ERR_UNSUPPORTED, "b200_effdet_postprocess: too many anchors per image for the rank table");
#define EF_LAUNCH(M)                                                                                                     \
  B200_CUDA(cudaFuncSetAttribute(effdet_nms_finalize_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2)); \
  effdet_nms_finalize_kernel<M><<<num_images, NMS_THREADS, smem2, stream>>>(np)
  NMS_DISPATCH_METRIC(metric, EF_LAUNCH)
#undef EF_LAUNCH
  B200_LAUNCH_CHECK();
  return B200_OK;
}

extern "C" size_t b200_effdet_postprocess_workspace_bytes(int num_levels, const int32_t* hw, int A, int num_images, int max_out) {
  int n_img = 0;
  for (int l = 0; l < num_levels; ++l) n_img += hw[2 * l] * hw[2 * l + 1] * A;
  return cand_layout(num_images, n_img, max_out, false, true).total;
}

// boxes: decoded boxes (the drop-in convert_outputs_one), or null with rel / table_dev given: decode inside the filter
// pass (convert_outputs_boxes + convert_outputs_one in one sweep; dec_out[l] receives the dense decoded tensor)
static int ef_post_impl(int num_levels, const int32_t* hw, int A, const float* table_dev, int C, int B, int first_image,
                        int num_images, const float* const boxes[], const float* const rel[], float* const dec_out[],
                        const float* const classes[], int max_out, float iou_thr, float score_thr, int metric, float* out_boxes,
                        long long* out_class_id, float* out_score, int32_t* out_sel_idx,
                        int32_t* out_sel_anchor, int32_t* out_count, void* workspace,
                        size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  EfFilterParams fp;
  B200_REQUIRE(hw && (boxes || (rel && table_dev)) && classes, B200_ERR_BAD_ARG, "b200_effdet_postprocess: null argument");
  const int n_img = ef_fill_levels(fp.lv, num_levels, hw, A, table_dev);
  B200_REQUIRE(n_img >= 0, B200_ERR_BAD_ARG, "b200_effdet_postprocess: bad level spec");
  B200_REQUIRE(C >= 1 && C <= 400, B200_ERR_UNSUPPORTED, "b200_effdet_postprocess: classes_num %d outside [1,400]", C);
  B200_REQUIRE(first_image >= 0 && num_images >= 0 && first_image + num_images <= B, B200_ERR_BAD_ARG, "b200_effdet_postprocess: image range outside the batch");
  B200_REQUIRE(metric >= B200_METRIC_EFF_IOU && metric <= B200_METRIC_EFF_CIOU, B200_ERR_BAD_ARG, "b200_effdet_postprocess: iou_type must be iou/giou/diou/ciou");
  B200_REQUIRE(max_out >= 1 && max_out <= NMS_MAX_OUT_LIMIT, B200_ERR_UNSUPPORTED, "b200_effdet_postprocess: max_out %d outside [1,%d]", max_out, NMS_MAX_OUT_LIMIT);
  if (num_images == 0) return B200_OK;
  B200_REQUIRE(out_boxes && out_class_id && out_score && out_count, B200_ERR_BAD_ARG, "b200_effdet_postprocess: null output");
  const CandLayout ws = cand_layout(num_images, n_img, max_out, false, true);
  B200_REQUIRE(workspace && workspace_bytes >= ws.total, B200_ERR_WORKSPACE, "b200_effdet_postprocess: workspace %zu < required %zu", workspace_bytes, ws.total);
  B200_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, B200_ERR_BAD_ARG, "b200_effdet_postprocess: workspace not 256-byte aligned");
  unsigned char* wsb = static_cast<unsigned char*>(workspace);
  fp.B0 = first_image; fp.NB = num_images; fp.C = C; fp.B = B;
  long long tb = 0;
  for (int l = 0; l < EF_MAX_LEVELS; ++l) {
    fp.tile_base[l] = tb;
    if (l < num_levels) {
      const float* bl = boxes ? boxes[l] : rel[l];
      B200_REQUIRE(bl && classes[l], B200_ERR_BAD_ARG, "b200_effdet_postprocess: null level %d", l);
      B200_REQUIRE(((reinterpret_cast<uintptr_t>(bl) | (dec_out && dec_out[l] ? reinterpret_cast<uintptr_t>(dec_out[l]) : 0)) & 15) == 0, B200_ERR_BAD_ARG,
                   "b200_effdet_postprocess: boxes level %d not 16-byte aligned", l);
      fp.cls[l] = classes[l];
      fp.boxes[l] = boxes ? reinterpret_cast<const float4*>(boxes[l]) : nullptr;
      fp.rel[l] = boxes ? nullptr : reinterpret_cast<const float4*>(rel[l]);
      fp.dec[l] = (!boxes && dec_out) ? reinterpret_cast<float4*>(dec_out[l]) : nullptr;
      tb += ((long long)num_images * fp.lv.anc_per_img[l] + 31) / 32;
    } else { fp.cls[l] = nullptr; fp.boxes[l] = nullptr; fp.rel[l] = nullptr; fp.dec[l] = nullptr; }
  }
  for (int l = num_levels; l <= EF_MAX_LEVELS; ++l) fp.tile_base[l] = tb;
  fp.st = cand_bind(ws, wsb, out_sel_idx != nullptr);
  B200_CUDA(cudaMemsetAsync(wsb, 0, ws.zeroed(out_sel_idx != nullptr), stream));
  using Ring = WarpSlabRing<EF_STAGES>;
  int warps = 8;
  while (warps > 1 && Ring::smem_bytes(warps, C) > 200 * 1024) warps >>= 1;
  const size_t smem1 = Ring::smem_bytes(warps, C);
  B200_CUDA(cudaFuncSetAttribute(effdet_filter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
  const int grid = Ring::grid(tb, warps, b200_sm_count());
  effdet_filter_kernel<<<grid, warps * 32, smem1, stream>>>(fp);
  B200_LAUNCH_CHECK();

  return ef_launch_nms(fp.st, num_images, max_out, iou_thr, score_thr, metric, out_boxes, out_class_id, out_score, out_sel_idx,
                       out_sel_anchor, out_count, stream);
}

extern "C" int b200_effdet_postprocess(int num_levels, const int32_t* hw, int A, int C, int B, int first_image,
                                       int num_images, const float* const boxes[], const float* const classes[],
                                       int max_out, float iou_thr, float score_thr, int metric, float* out_boxes,
                                       long long* out_class_id, float* out_score, int32_t* out_sel_idx,
                                       int32_t* out_sel_anchor, int32_t* out_count, void* workspace,
                                       size_t workspace_bytes, void* stream_) {
  B200_REQUIRE(boxes, B200_ERR_BAD_ARG, "b200_effdet_postprocess: null argument");
  return ef_post_impl(num_levels, hw, A, nullptr, C, B, first_image, num_images, boxes, nullptr, nullptr, classes, max_out, iou_thr,
                      score_thr, metric, out_boxes, out_class_id, out_score, out_sel_idx, out_sel_anchor, out_count, workspace,
                      workspace_bytes, stream_);
}

// CTAs of 256 anchors per (level, image); returns the grid size
static int ef_assign_plan(EfAssignParams& p) {
  int cta = 0;
  for (int l = 0; l < EF_MAX_LEVELS; ++l) {
    p.cta_base[l] = cta;
    p.chunks_per_img[l] = l < p.lv.num_levels ? (p.lv.anc_per_img[l] + 255) / 256 : 1;
    if (l < p.lv.num_levels) cta += p.chunks_per_img[l] * p.B;
  }
  p.cta_base[EF_MAX_LEVELS] = cta;
  return cta;
}

static int ef_assign_impl(int num_levels, const int32_t* hw, int A, const float* table_dev, int C, int B,
                          const float* gt_boxes, const int32_t* gt_classes, const int32_t* gt_offsets, float iou_thr,
                          float* const out_boxes[], float* const out_onehot[], int32_t* const out_class[],
                          unsigned char* const out_mask[], void* stream) {
  EfAssignParams p;
  B200_REQUIRE(hw && table_dev && gt_offsets && out_boxes && (out_onehot || out_class) && out_mask, B200_ERR_BAD_ARG, "b200_effdet_assign_targets: null argument");
  B200_REQUIRE(ef_fill_levels(p.lv, num_levels, hw, A, table_dev) >= 0, B200_ERR_BAD_ARG, "b200_effdet_assign_targets: bad level spec");
  B200_REQUIRE(B >= 0 && C >= 1, B200_ERR_BAD_ARG, "b200_effdet_assign_targets: bad sizes");
  if (B == 0) return B200_OK;
  p.B = B; p.C = C; p.thr = iou_thr;
  p.magic_c = C == 1 ? 0u : (uint32_t)((1ull << 32) / (unsigned long long)C + 1ull);
  p.gt_boxes = gt_boxes; p.gt_classes = gt_classes; p.gt_offsets = gt_offsets;
  p.out_match = nullptr; p.positives = nullptr;
  for (int l = 0; l < EF_MAX_LEVELS; ++l) {
    if (l < num_levels) {
      B200_REQUIRE(out_boxes[l] && (out_onehot ? out_onehot[l] != nullptr : out_class[l] != nullptr) && out_mask[l], B200_ERR_BAD_ARG,
                   "b200_effdet_assign_targets: null level %d", l);
      B200_REQUIRE((reinterpret_cast<uintptr_t>(out_boxes[l]) & 15) == 0, B200_ERR_BAD_ARG, "b200_effdet_assign_targets: out_boxes level %d not 16-byte aligned", l);
      p.out_boxes[l] = reinterpret_cast<float4*>(out_boxes[l]);
      p.out_onehot[l] = out_onehot ? out_onehot[l] : nullptr;
      p.out_class[l] = out_onehot ? nullptr : out_class[l];
      p.out_mask[l] = out_mask[l];
    } else { p.out_boxes[l] = nullptr; p.out_onehot[l] = nullptr; p.out_class[l] = nullptr; p.out_mask[l] = nullptr; }
  }
  const int cta = ef_assign_plan(p);
  effdet_assign_kernel<<<cta, 256, 0, (cudaStream_t)stream>>>(p);
  B200_LAUNCH_CHECK();
  return B200_OK;
}

extern "C" int b200_effdet_assign_targets(int num_levels, const int32_t* hw, int A, const float* table_dev, int C, int B,
                                          const float* gt_boxes, const int32_t* gt_classes, const int32_t* gt_offsets,
                                          float iou_thr, float* const out_boxes[], float* const out_onehot[],
                                          unsigned char* const out_mask[], void* stream) {
  B200_REQUIRE(out_onehot, B200_ERR_BAD_ARG, "b200_effdet_assign_targets: null argument");
  return ef_assign_impl(num_levels, hw, A, table_dev, C, B, gt_boxes, gt_classes, gt_offsets, iou_thr, out_boxes, out_onehot,
                        nullptr, out_mask, stream);
}

extern "C" int b200_effdet_assign_targets_indexed(int num_levels, const int32_t* hw, int A, const float* table_dev, int C, int B,
                                                  const float* gt_boxes, const int32_t* gt_classes, const int32_t* gt_offsets,
                                                  float iou_thr, float* const out_boxes[], int32_t* const out_class[],
                                                  unsigned char* const out_mask[], void* stream) {
  B200_REQUIRE(out_class, B200_ERR_BAD_ARG, "b200_effdet_assign_targets_indexed: null argument");
  return ef_assign_impl(num_levels, hw, A, table_dev, C, B, gt_boxes, gt_classes, gt_offsets, iou_thr, out_boxes, nullptr,
                        out_class, out_mask, stream);
}

// Stage 1 of the loss from box lists (effdet_loss.cu has stage 2): the anchor -> GT row of every anchor of the batch
// into the workspace, sums zeroed and sums[2L] = this call's matched anchors.  The IoU, the culling, the tie rule and the
// threshold are generate_targets' own (the same kernel in match mode).
size_t efb_workspace_bytes(int num_levels, int anchors_per_image, int B);   // effdet_loss.cu

extern "C" int b200_effdet_loss_from_boxes_match(int num_levels, const int32_t* hw, int A, const float* table_dev, int B,
                                                 const float* gt_boxes, const int32_t* gt_offsets, int total_boxes,
                                                 float iou_thr, double* sums, void* workspace, size_t workspace_bytes,
                                                 void* stream) {
  const char* who = "b200_effdet_loss_from_boxes_match";
  EfAssignParams p;
  B200_REQUIRE(hw && table_dev && gt_offsets && sums, B200_ERR_BAD_ARG, "%s: null argument", who);
  const int n_img = ef_fill_levels(p.lv, num_levels, hw, A, table_dev);
  B200_REQUIRE(n_img >= 0, B200_ERR_BAD_ARG, "%s: bad level spec", who);
  B200_REQUIRE(B >= 0 && total_boxes >= 0, B200_ERR_BAD_ARG, "%s: negative batch or box count", who);
  B200_REQUIRE(total_boxes == 0 || gt_boxes, B200_ERR_BAD_ARG, "%s: null gt_boxes", who);
  const size_t need = efb_workspace_bytes(num_levels, n_img, B);
  B200_REQUIRE(workspace && workspace_bytes >= need, B200_ERR_WORKSPACE, "%s: workspace %zu < required %zu", who, workspace_bytes, need);
  B200_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, B200_ERR_BAD_ARG, "%s: workspace not 256-byte aligned", who);
  B200_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * (2 * num_levels + 1), (cudaStream_t)stream));
  if (B == 0) return B200_OK;
  p.B = B; p.C = 1; p.magic_c = 0u; p.thr = iou_thr;
  p.gt_boxes = gt_boxes; p.gt_classes = nullptr; p.gt_offsets = gt_offsets;
  for (int l = 0; l < EF_MAX_LEVELS; ++l) { p.out_boxes[l] = nullptr; p.out_onehot[l] = nullptr; p.out_class[l] = nullptr; p.out_mask[l] = nullptr; }
  p.out_match = static_cast<int32_t*>(workspace);
  p.positives = sums + 2 * num_levels;
  const int cta = ef_assign_plan(p);
  effdet_assign_kernel<<<cta, 256, 0, (cudaStream_t)stream>>>(p);
  B200_LAUNCH_CHECK();
  return B200_OK;
}

// ---- fused eval-step stream (test_step, efficientnet/efficientdet_net_train.py:135-169) ----------------------------
// The reference's test_step reads the class logits twice: FocalLoss (:150) and, after convert_outputs_boxes (:153), the
// per-image argmax / max of convert_outputs_one (anchors.py:172-174).  Here ONE pass over every level does
//   * focal loss of the tile's logits against the one-hot targets (flat 128-bit streaming loads, both tensors),
//   * argmax / max over each anchor's C logits (the tile also goes to shared memory; four lanes per anchor),
//   * box decode from the head offsets and the anchor table (anchors.py:245-274) -> the dense decoded tensor,
//   * Huber box loss + positive count (box_loss.py:17-29), and
//   * the append of every non-background anchor to its image's candidate list (anchors.py:179-189).
// (Without targets — convert_outputs_boxes + convert_outputs_one alone — the per-warp bulk-copy filter above is the faster
// stream and takes the decode along: b200_effdet_decode_postprocess.)
#define EFU_TILE 64      // anchors per tile
#define EFU_THREADS 256

struct EfFusedParams {
  EfLevels lv;
  int B, C;
  const float* cls[EF_MAX_LEVELS];        // (B,H,W,A,C) logits
  const float* cls_true[EF_MAX_LEVELS];   // (B,H,W,A,C) targets
  const float4* rel[EF_MAX_LEVELS];       // (B,H,W,A,4) head offsets ty,tx,th,tw
  const float4* box_true[EF_MAX_LEVELS];
  const unsigned char* mask[EF_MAX_LEVELS];
  float4* dec[EF_MAX_LEVELS];             // decoded boxes out
  long long tile_base[EF_MAX_LEVELS + 1];
  CandStore st;
  float alpha, gamma, delta, label_smoothing;
  double* partials;                       // [gridDim.x][num_levels][3] focal, huber, positives
};

// Warp roles inside a CTA (tile = 64 anchors):
//   warps 2-7 (CLASS stream, 192 threads): the tile's logits (and one-hot targets) arrive in shared memory by 1-D bulk
//     asynchronous copies (bulkcopy.cuh; two stages: the copy of the CTA's next tile is in flight while this one is
//     processed); focal terms from flat 128-bit shared-memory reads, then the per-anchor argmax with three lanes
//     per anchor (partial (max, first index) per third of the C logits -> shared memory);
//   warps 0-1 (BOX half, lane <-> anchor): head offsets / box targets / mask straight from global memory, decode, Huber,
//     and — behind the tile's single CTA barrier — the fold of the three argmax partials and the candidate append.
// Both halves are ~600-800 instructions per warp and tile and independent, so they run side by side.
#define EFU_BOX_WARPS 2
#define EFU_STREAM_THREADS (EFU_THREADS - 32 * EFU_BOX_WARPS)
#define EFU_STAGES 2

template <bool G15>
__global__ void __launch_bounds__(EFU_THREADS, 2) effdet_stream_kernel(EfFusedParams p) {
  extern __shared__ __align__(128) unsigned char efu_smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int C = p.C;
  const uint32_t tile_bytes = (uint32_t)EFU_TILE * (uint32_t)C * 4u;
  // stage s: [x tile][y tile]
  const uint32_t stage_bytes = tile_bytes * 2u;
  __shared__ __align__(8) uint64_t s_bar[EFU_STAGES];
  __shared__ double s_part[EF_MAX_LEVELS][3];
  __shared__ double s_red[EFU_THREADS / 32][3];
  __shared__ float s_m[2][EFU_TILE][3];
  __shared__ int s_mi[2][EFU_TILE][3];
  if (tid < EF_MAX_LEVELS * 3) s_part[tid / 3][tid % 3] = 0.0;
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < EFU_STAGES; ++s) bc_mbar_init(&s_bar[s], 1);
    bc_fence_mbar_init();
  }
  __syncthreads();
  const long long n_tiles = p.tile_base[p.lv.num_levels];
  double focal = 0.0;
  float hub = 0.f;
  unsigned int pos = 0;
  int cur_level = -1;
  auto flush = [&](int level) {   // block-reduce this thread's running sums into the level's slot
    double v0 = warp_sum_d(focal), v1 = warp_sum_d((double)hub), v2 = warp_sum_d((double)pos);
    if (lane == 0) { s_red[warp][0] = v0; s_red[warp][1] = v1; s_red[warp][2] = v2; }
    __syncthreads();
    if (tid < 3) {
      double sacc = 0.0;
      for (int w = 0; w < EFU_THREADS / 32; ++w) sacc += s_red[w][tid];
      s_part[level][tid] += sacc;
    }
    __syncthreads();
    focal = 0.0; hub = 0.f; pos = 0;
  };
  // (level, first anchor, anchors, bulk-copyable) of a tile
  auto locate = [&](long long t, int& l, long long& rec0, int& nrec) {
    l = 0;
#pragma unroll
    for (int k = 1; k < EF_MAX_LEVELS; ++k) if (k < p.lv.num_levels && t >= p.tile_base[k]) l = k;
    rec0 = (t - p.tile_base[l]) * EFU_TILE;
    const long long remain = (long long)p.B * p.lv.anc_per_img[l] - rec0;
    nrec = remain < EFU_TILE ? (int)remain : EFU_TILE;
  };
  auto bulk_ok = [&](int l, long long rec0, int nrec) {
    const uintptr_t ax = reinterpret_cast<uintptr_t>(p.cls[l] + rec0 * C);
    const uintptr_t ay = reinterpret_cast<uintptr_t>(p.cls_true[l] + rec0 * C);
    return (((ax | ay) & 15) == 0) && ((((uint32_t)nrec * (uint32_t)C * 4u) & 15u) == 0u);
  };
  auto issue = [&](long long t, int s) {   // one thread: start the copies of tile t into stage s
    int l, nrec; long long rec0;
    locate(t, l, rec0, nrec);
    if (!bulk_ok(l, rec0, nrec)) return;   // ragged / unaligned tile: read straight from global memory when it is consumed
    const uint32_t bytes = (uint32_t)nrec * (uint32_t)C * 4u;
    unsigned char* dst = efu_smem + (size_t)s * stage_bytes;
    bc_fence_proxy_async();
    bc_mbar_expect_tx(&s_bar[s], bytes * 2u);
    bc_bulk_g2s(dst, p.cls[l] + rec0 * C, bytes, &s_bar[s]);
    bc_bulk_g2s(dst + tile_bytes, p.cls_true[l] + rec0 * C, bytes, &s_bar[s]);
  };
  const bool box_warp = warp < EFU_BOX_WARPS;
  const int st = tid - 32 * EFU_BOX_WARPS;   // index among the stream threads
  const int q3 = (C + 2) / 3;
  if (tid == 32 * EFU_BOX_WARPS) {
#pragma unroll
    for (int s = 0; s < EFU_STAGES; ++s) {
      const long long t = (long long)blockIdx.x + (long long)s * gridDim.x;
      if (t < n_tiles) issue(t, s);
    }
  }
  uint32_t phase_bits = 0;   // parity of each stage's barrier
  int j = 0;
  for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x, ++j) {
    const int s = j & (EFU_STAGES - 1), pb = j & 1;
    int l, nrec; long long rec0;
    locate(t, l, rec0, nrec);
    if (l != cur_level) {
      if (cur_level >= 0) flush(cur_level);
      cur_level = l;
    }
    const int api = p.lv.anc_per_img[l];
    const long long total = (long long)p.B * api;
    const bool bulk = bulk_ok(l, rec0, nrec);
    int img = 0;
    uint32_t aidx = 0;
    float4 d4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (box_warp) {
      // ---- box half: lane <-> anchor ----
      if (tid < nrec) {
        const long long rec = rec0 + tid;
        const float4 r4 = __ldcs(p.rel[l] + rec);
        const float4 t4 = __ldcs(p.box_true[l] + rec);
        const unsigned char mk = p.mask[l][rec];
        int rin;
        if (total < 0x7fffffffLL) { img = (int)((uint32_t)rec / (uint32_t)api); rin = (int)((uint32_t)rec - (uint32_t)img * (uint32_t)api); }
        else { img = (int)(rec / api); rin = (int)(rec - (long long)img * api); }
        int y, x, an_i;
        ef_split(p.lv, l, rin, y, x, an_i);
        d4 = ef_decode_box(ef_anchor(p.lv, l, y, x, an_i), r4);
        if (p.dec[l]) __stcs(p.dec[l] + rec, d4);
        hub += el_huber(t4.x, r4.x, p.delta) + el_huber(t4.y, r4.y, p.delta) + el_huber(t4.z, r4.z, p.delta) + el_huber(t4.w, r4.w, p.delta);
        pos += mk ? 1u : 0u;
        aidx = (uint32_t)(p.lv.anchor_base[l] + rin);
      }
    } else {
      // ---- class stream ----
      float* xs = reinterpret_cast<float*>(efu_smem + (size_t)s * stage_bytes);
      const float* ys = reinterpret_cast<const float*>(efu_smem + (size_t)s * stage_bytes + tile_bytes);
      const int n_el = nrec * C;
      float f0 = 0.f, f1 = 0.f;
      if (bulk) {
        bc_mbar_wait(&s_bar[s], (phase_bits >> s) & 1u);
        const int n_vec = n_el >> 2;
#pragma unroll 2
        for (int i = st; i < n_vec; i += EFU_STREAM_THREADS) {
          const float4 x = reinterpret_cast<const float4*>(xs)[i];
          const float4 y = reinterpret_cast<const float4*>(ys)[i];
          f0 += el_focal<G15>(y.x, x.x, p.alpha, p.gamma, p.label_smoothing) + el_focal<G15>(y.y, x.y, p.alpha, p.gamma, p.label_smoothing);
          f1 += el_focal<G15>(y.z, x.z, p.alpha, p.gamma, p.label_smoothing) + el_focal<G15>(y.w, x.w, p.alpha, p.gamma, p.label_smoothing);
        }
      } else {
        // ragged tail of a level or an unaligned tensor: plain loads; the logits still go to the stage for the argmax
        const float* xg = p.cls[l] + rec0 * C;
        const float* yg = p.cls_true[l] + rec0 * C;
        for (int e = st; e < n_el; e += EFU_STREAM_THREADS) {
          const float xv = __ldg(xg + e);
          xs[e] = xv;
          f0 += el_focal<G15>(__ldg(yg + e), xv, p.alpha, p.gamma, p.label_smoothing);
        }
        asm volatile("bar.sync 1, %0;" ::"n"(EFU_STREAM_THREADS) : "memory");   // stream warps only: the tile is complete
      }
      focal += (double)f0 + (double)f1;
      // per-anchor argmax, three lanes per anchor: tf.argmax (first maximal index) / reduce_max over a third of the C
      // logits each; the box warps fold the three partials in ascending index order
      const int a = st / 3, part = st - a * 3;
      float m = -INFINITY;
      int mi = -1;
      if (a < nrec) {
        const float* r = xs + a * C;
        const int c0 = part * q3, c1 = min(C, c0 + q3);
        int c = c0;
        if (part == 0) { m = r[0]; mi = 0; c = 1; }   // the scan starts from element 0 exactly as a serial one (NaN there sticks)
        for (; c + 4 <= c1; c += 4) {                  // loads first, then the dependent compare / select chain
          const float v0 = r[c], v1 = r[c + 1], v2 = r[c + 2], v3 = r[c + 3];
          if (v0 > m) { m = v0; mi = c; }
          if (v1 > m) { m = v1; mi = c + 1; }
          if (v2 > m) { m = v2; mi = c + 2; }
          if (v3 > m) { m = v3; mi = c + 3; }
        }
        for (; c < c1; ++c) { const float v = r[c]; if (v > m) { m = v; mi = c; } }
      }
      s_m[pb][a][part] = m;
      s_mi[pb][a][part] = mi;
    }
    __syncthreads();   // the tile's single CTA barrier: the stage is consumed, the argmax partials are published
    if (bulk) phase_bits ^= (1u << s);
    if (tid == 32 * EFU_BOX_WARPS) {
      const long long tn = t + (long long)EFU_STAGES * gridDim.x;
      if (tn < n_tiles) issue(tn, s);
    }
    if (box_warp) {
      // ---- fold the partials, candidate append (anc:179-189), one atomic per (warp, image) ----
      float m = s_m[pb][tid][0];
      int mi = s_mi[pb][tid][0];
#pragma unroll
      for (int k = 1; k < 3; ++k) { const float vk = s_m[pb][tid][k]; if (vk > m) { m = vk; mi = s_mi[pb][tid][k]; } }
      const bool pass = (tid < nrec) && (mi != 0);   // classes_mask = classes_id != 0 (anc:179)
      warp_append_by_image(p.st, pass, img, aidx, [&](size_t slot) {
        p.st.box[slot] = d4; p.st.score[slot] = m; p.st.cls[slot] = mi;
      });
    }
    // the partial buffers alternate by tile parity: the stream warps write buffer pb again only two tiles later, behind
    // the next tile's barrier, which the box warps reach after this append
  }
  if (cur_level >= 0) flush(cur_level);
  __syncthreads();
  if (tid < p.lv.num_levels * 3)
    p.partials[((size_t)blockIdx.x * p.lv.num_levels + tid / 3) * 3 + tid % 3] = s_part[tid / 3][tid % 3];
}

// sums layout of effdet_loss.cu: [0..L) focal_l, [L..2L) huber_l, [2L] positives
__global__ void __launch_bounds__(256) effdet_stream_reduce_kernel(const double* __restrict__ partials, int n_cta, int L, double* __restrict__ sums) {
  __shared__ double s_red[8][3];
  const int l = blockIdx.x;
  double a[3] = {0.0, 0.0, 0.0};
  for (int c = threadIdx.x; c < n_cta; c += 256) {
    const double* q = partials + ((size_t)c * L + l) * 3;
    a[0] += q[0]; a[1] += q[1]; a[2] += q[2];
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 3; ++k) { const double v = warp_sum_d(a[k]); if (lane == 0) s_red[warp][k] = v; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double sacc[3] = {0.0, 0.0, 0.0};
    for (int w = 0; w < 8; ++w) for (int k = 0; k < 3; ++k) sacc[k] += s_red[w][k];
    sums[l] = sacc[0];
    sums[L + l] = sacc[1];
    atomicAdd(&sums[2 * L], sacc[2]);  // integer-valued: exact and order-independent
  }
}

#define EFU_GRID_PER_SM 16

static size_t efu_partials_bytes(int num_levels) {
  return b200_align_up(sizeof(double) * 3 * (size_t)num_levels * (size_t)b200_sm_count() * EFU_GRID_PER_SM, 256);
}

extern "C" size_t b200_effdet_eval_workspace_bytes(int num_levels, const int32_t* hw, int A, int num_images, int max_out) {
  return b200_effdet_postprocess_workspace_bytes(num_levels, hw, A, num_images, max_out) + efu_partials_bytes(num_levels);
}

static int efu_impl(int num_levels, const int32_t* hw, int A, const float* table_dev, int C, int B,
                    const float* const true_boxes[], const float* const true_classes[], const unsigned char* const true_masks[],
                    const float* const pred_boxes[], const float* const pred_classes[], float alpha, float gamma, float delta,
                    float label_smoothing, double* sums_out, float* const out_decoded[], int max_out, float iou_thr,
                    float score_thr, int metric, float* out_boxes, long long* out_class_id, float* out_score,
                    int32_t* out_sel_idx, int32_t* out_sel_anchor, int32_t* out_count, void* workspace, size_t workspace_bytes,
                    void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  const char* who = "b200_effdet_eval_step";
  EfFusedParams p;
  B200_REQUIRE(hw && table_dev && pred_boxes && pred_classes, B200_ERR_BAD_ARG, "%s: null argument", who);
  B200_REQUIRE(true_boxes && true_classes && true_masks && sums_out, B200_ERR_BAD_ARG, "%s: null target argument", who);
  const int n_img = ef_fill_levels(p.lv, num_levels, hw, A, table_dev);
  B200_REQUIRE(n_img >= 0, B200_ERR_BAD_ARG, "%s: bad level spec", who);
  B200_REQUIRE(C >= 1 && C <= 400, B200_ERR_UNSUPPORTED, "%s: classes_num %d outside [1,400]", who, C);
  B200_REQUIRE(B >= 0, B200_ERR_BAD_ARG, "%s: negative batch", who);
  B200_REQUIRE(metric >= B200_METRIC_EFF_IOU && metric <= B200_METRIC_EFF_CIOU, B200_ERR_BAD_ARG, "%s: iou_type must be iou/giou/diou/ciou", who);
  B200_REQUIRE(max_out >= 1 && max_out <= NMS_MAX_OUT_LIMIT, B200_ERR_UNSUPPORTED, "%s: max_out %d outside [1,%d]", who, max_out, NMS_MAX_OUT_LIMIT);
  if (B == 0) return B200_OK;
  B200_REQUIRE(out_boxes && out_class_id && out_score && out_count, B200_ERR_BAD_ARG, "%s: null output", who);
  const CandLayout ws = cand_layout(B, n_img, max_out, false, true);
  const size_t part_bytes = efu_partials_bytes(num_levels);
  B200_REQUIRE(workspace && workspace_bytes >= ws.total + part_bytes, B200_ERR_WORKSPACE, "%s: workspace %zu < required %zu", who, workspace_bytes, ws.total + part_bytes);
  B200_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, B200_ERR_BAD_ARG, "%s: workspace not 256-byte aligned", who);
  unsigned char* wsb = static_cast<unsigned char*>(workspace);
  p.B = B; p.C = C;
  long long tb = 0;
  for (int l = 0; l < EF_MAX_LEVELS; ++l) {
    p.tile_base[l] = tb;
    p.cls[l] = nullptr; p.cls_true[l] = nullptr; p.rel[l] = nullptr; p.box_true[l] = nullptr; p.mask[l] = nullptr; p.dec[l] = nullptr;
    if (l >= num_levels) continue;
    B200_REQUIRE(pred_boxes[l] && pred_classes[l], B200_ERR_BAD_ARG, "%s: null level %d", who, l);
    B200_REQUIRE(true_boxes[l] && true_classes[l] && true_masks[l], B200_ERR_BAD_ARG, "%s: null target level %d", who, l);
    const uintptr_t al = reinterpret_cast<uintptr_t>(pred_boxes[l]) | reinterpret_cast<uintptr_t>(true_boxes[l]) |
                         (out_decoded && out_decoded[l] ? reinterpret_cast<uintptr_t>(out_decoded[l]) : 0);
    B200_REQUIRE((al & 15) == 0, B200_ERR_BAD_ARG, "%s: box tensors of level %d must be 16-byte aligned", who, l);
    p.cls[l] = pred_classes[l];
    p.rel[l] = reinterpret_cast<const float4*>(pred_boxes[l]);
    p.dec[l] = out_decoded ? reinterpret_cast<float4*>(out_decoded[l]) : nullptr;
    p.cls_true[l] = true_classes[l];
    p.box_true[l] = reinterpret_cast<const float4*>(true_boxes[l]);
    p.mask[l] = true_masks[l];
    tb += ((long long)B * p.lv.anc_per_img[l] + EFU_TILE - 1) / EFU_TILE;
  }
  for (int l = num_levels; l <= EF_MAX_LEVELS; ++l) p.tile_base[l] = tb;
  p.st = cand_bind(ws, wsb, out_sel_idx != nullptr);
  p.alpha = alpha; p.gamma = gamma; p.delta = delta; p.label_smoothing = label_smoothing;
  p.partials = reinterpret_cast<double*>(wsb + ws.total);
  B200_CUDA(cudaMemsetAsync(wsb, 0, ws.zeroed(out_sel_idx != nullptr), stream));
  B200_REQUIRE(C <= 128, B200_ERR_UNSUPPORTED, "%s: the fused pass stages %d-anchor tiles in shared memory: classes_num %d > 128 (use the separate calls)", who, EFU_TILE, C);
  const size_t smem = (size_t)EFU_STAGES * EFU_TILE * C * sizeof(float) * 2;
  long long want = tb;
  const long long cap = (long long)b200_sm_count() * EFU_GRID_PER_SM;
  const int grid = (int)(want < cap ? (want < 1 ? 1 : want) : cap);
#define EFU_LAUNCH(G)                                                                                                   \
  do {                                                                                                                  \
    B200_CUDA(cudaFuncSetAttribute(effdet_stream_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    effdet_stream_kernel<G><<<grid, EFU_THREADS, smem, stream>>>(p);                                                  \
  } while (0)
  if (gamma == 1.5f) EFU_LAUNCH(true);
  else EFU_LAUNCH(false);
#undef EFU_LAUNCH
  B200_LAUNCH_CHECK();
  B200_CUDA(cudaMemsetAsync(sums_out, 0, sizeof(double) * (2 * num_levels + 1), stream));
  effdet_stream_reduce_kernel<<<num_levels, 256, 0, stream>>>(p.partials, grid, num_levels, sums_out);
  B200_LAUNCH_CHECK();
  return ef_launch_nms(p.st, B, max_out, iou_thr, score_thr, metric, out_boxes, out_class_id, out_score, out_sel_idx, out_sel_anchor,
                       out_count, stream);
}

// test_step in one call: sums_out [2L+1] fp64 (un-normalised focal_l, huber_l, positives: feed b200_focal_box_finalize or
// its _dp form), out_decoded[l] = convert_outputs_boxes, then convert_outputs_one for every image of the batch.
extern "C" int b200_effdet_eval_step(int num_levels, const int32_t* hw, int A, const float* table_dev, int C, int B,
                                     const float* const true_boxes[], const float* const true_classes[],
                                     const unsigned char* const true_masks[], const float* const pred_boxes[],
                                     const float* const pred_classes[], float alpha, float gamma, float delta,
                                     float label_smoothing, double* sums_out, float* const out_decoded[], int max_out,
                                     float iou_thr, float score_thr, int metric, float* out_boxes, long long* out_class_id,
                                     float* out_score, int32_t* out_sel_idx, int32_t* out_sel_anchor, int32_t* out_count,
                                     void* workspace, size_t workspace_bytes, void* stream) {
  return efu_impl(num_levels, hw, A, table_dev, C, B, true_boxes, true_classes, true_masks, pred_boxes, pred_classes, alpha,
                  gamma, delta, label_smoothing, sums_out, out_decoded, max_out, iou_thr, score_thr, metric, out_boxes, out_class_id,
                  out_score, out_sel_idx, out_sel_anchor, out_count, workspace, workspace_bytes, stream);
}

// convert_outputs_boxes + convert_outputs_one of the whole batch in one pass over the heads (no targets, no loss).
extern "C" int b200_effdet_decode_postprocess(int num_levels, const int32_t* hw, int A, const float* table_dev, int C, int B,
                                              const float* const pred_boxes[], const float* const pred_classes[],
                                              float* const out_decoded[], int max_out, float iou_thr, float score_thr, int metric,
                                              float* out_boxes, long long* out_class_id, float* out_score, int32_t* out_sel_idx,
                                              int32_t* out_sel_anchor, int32_t* out_count, void* workspace, size_t workspace_bytes,
                                              void* stream) {
  // without targets the per-warp bulk-copy filter (lane <-> anchor, no CTA barriers) is the faster stream: the decode rides
  // on it (one coalesced 16-byte load and store per lane); the CTA-tiled kernel above pays off only with the focal terms
  B200_REQUIRE(pred_boxes && table_dev, B200_ERR_BAD_ARG, "b200_effdet_decode_postprocess: null argument");
  return ef_post_impl(num_levels, hw, A, table_dev, C, B, 0, B, nullptr, pred_boxes, out_decoded, pred_classes, max_out, iou_thr,
                      score_thr, metric, out_boxes, out_class_id, out_score, out_sel_idx, out_sel_anchor, out_count, workspace,
                      workspace_bytes, stream);
}
