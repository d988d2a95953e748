// unletterbox.cu — the box post-processing of the serving path (SURVEY §8f N4, the part that has a closed form):
// views/object_detection.py:70-85 maps the boxes Predict returns on the letterboxed image back to the original
// image, clips them, drops boxes not larger than 2 px and truncates to int32.  (The letterbox itself: letterbox.cu.)
//
//   x' = ((x * W_in - pad_left) / (W_in - pad_left - pad_right)) * W_old      (fp32 step by step, NumPy 1.x casting:
//   y' = ((y * H_in - pad_top ) / (H_in - pad_top  - pad_bottom)) * H_old       float32 array (op) integer scalar -> float32)
//   x1,y1 < 0 -> 0;  x2 > W_old -> W_old;  y2 > H_old -> H_old;  keep (x2 - x1 > 2) and (y2 - y1 > 2);  int32 truncation
//
// One CTA per image, one thread per row; kept rows are compacted in order (ballot prefix).  The padding and original
// size are either one set for the whole batch (b200_unletterbox_boxes) or read per image from a device array
// (b200_unletterbox_boxes_batch: frames of different sizes in one launch).
#include "detmath.h"
#include "common.cuh"

struct UlbParams {
  const float4* boxes;      // [B, max_rows] normalised x1,y1,x2,y2 on the letterboxed image
  const int32_t* counts;    // [B] valid rows per image, or nullptr (= max_rows)
  int B, max_rows;
  float in_w, in_h, pad_top, pad_bottom, pad_left, pad_right, old_w, old_h;
  const int32_t* geometry;  // [B, 6] top, bottom, left, right, old_w, old_h per image, or nullptr (= the scalars above)
  int4* out_boxes;          // [B, max_rows] int32 x1,y1,x2,y2 (kept rows first)
  int32_t* out_index;       // [B, max_rows] source row of every kept row
  int32_t* out_count;       // [B]
};

__global__ void __launch_bounds__(256) unletterbox_kernel(UlbParams p) {
  __shared__ int s_warp[8];
  __shared__ int s_base;
  const int img = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n = p.counts ? min(p.counts[img], p.max_rows) : p.max_rows;
  float pad_top = p.pad_top, pad_bottom = p.pad_bottom, pad_left = p.pad_left, pad_right = p.pad_right, old_w = p.old_w, old_h = p.old_h;
  if (p.geometry) {
    const int32_t* g = p.geometry + (size_t)img * 6;
    pad_top = (float)g[0]; pad_bottom = (float)g[1]; pad_left = (float)g[2]; pad_right = (float)g[3];
    old_w = (float)g[4]; old_h = (float)g[5];
  }
  const float den_x = DM_SUB(DM_SUB(p.in_w, pad_left), pad_right), den_y = DM_SUB(DM_SUB(p.in_h, pad_top), pad_bottom);
  if (threadIdx.x == 0) s_base = 0;
  __syncthreads();
  for (int r0 = 0; r0 < n; r0 += 256) {
    const int r = r0 + (int)threadIdx.x;
    bool keep = false;
    float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < n) {
      b = p.boxes[(size_t)img * p.max_rows + r];
      b.x = DM_MUL(DM_DIV(DM_SUB(DM_MUL(b.x, p.in_w), pad_left), den_x), old_w);
      b.z = DM_MUL(DM_DIV(DM_SUB(DM_MUL(b.z, p.in_w), pad_left), den_x), old_w);
      b.y = DM_MUL(DM_DIV(DM_SUB(DM_MUL(b.y, p.in_h), pad_top), den_y), old_h);
      b.w = DM_MUL(DM_DIV(DM_SUB(DM_MUL(b.w, p.in_h), pad_top), den_y), old_h);
      if (b.x < 0.0f) b.x = 0.0f;            // y_boxes[:,0][y_boxes[:,0]<0] = 0 (NaN stays)
      if (b.y < 0.0f) b.y = 0.0f;
      if (b.z > old_w) b.z = old_w;
      if (b.w > old_h) b.w = old_h;
      keep = (DM_SUB(b.z, b.x) > 2.0f) && (DM_SUB(b.w, b.y) > 2.0f);
    }
    const uint32_t bits = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) s_warp[warp] = __popc(bits);
    __syncthreads();
    int before = s_base;
    for (int w = 0; w < warp; ++w) before += s_warp[w];
    if (keep) {
      const size_t slot = (size_t)img * p.max_rows + before + __popc(bits & ((1u << lane) - 1u));
      p.out_boxes[slot] = make_int4((int)b.x, (int)b.y, (int)b.z, (int)b.w);  // astype(np.int32): truncation
      p.out_index[slot] = r;
    }
    __syncthreads();
    if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < 8; ++w) t += s_warp[w]; s_base += t; }
    __syncthreads();
  }
  if (threadIdx.x == 0) p.out_count[img] = s_base;
}

// Checks shared by both entry points; `p` carries the geometry, the rest is filled in here.
static int ulb_launch(const char* who, UlbParams& p, const float* boxes, const int32_t* counts, int B, int max_rows,
                      const int32_t image_size[2], int32_t* out_boxes, int32_t* out_index, int32_t* out_count, void* stream) {
  B200_REQUIRE(B >= 0 && max_rows >= 0, B200_ERR_BAD_ARG, "%s: bad sizes", who);
  if (B == 0) return B200_OK;
  B200_REQUIRE(image_size && out_count, B200_ERR_BAD_ARG, "%s: null argument", who);
  B200_REQUIRE(max_rows == 0 || (boxes && out_boxes && out_index), B200_ERR_BAD_ARG, "%s: null buffer", who);
  B200_REQUIRE(((reinterpret_cast<uintptr_t>(boxes) | reinterpret_cast<uintptr_t>(out_boxes)) & 15) == 0, B200_ERR_BAD_ARG,
               "%s: boxes / out_boxes not 16-byte aligned", who);
  p.boxes = reinterpret_cast<const float4*>(boxes); p.counts = counts; p.B = B; p.max_rows = max_rows;
  p.in_w = (float)image_size[0]; p.in_h = (float)image_size[1];
  p.out_boxes = reinterpret_cast<int4*>(out_boxes); p.out_index = out_index; p.out_count = out_count;
  unletterbox_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(p);
  B200_LAUNCH_CHECK();
  return B200_OK;
}

extern "C" int b200_unletterbox_boxes(const float* boxes, const int32_t* counts, int B, int max_rows, const int32_t image_size[2],
                                      const int32_t padding[4], const int32_t image_size_old[2], int32_t* out_boxes,
                                      int32_t* out_index, int32_t* out_count, void* stream) {
  B200_REQUIRE(B >= 0 && max_rows >= 0, B200_ERR_BAD_ARG, "b200_unletterbox_boxes: bad sizes");
  if (B == 0) return B200_OK;
  B200_REQUIRE(padding && image_size_old, B200_ERR_BAD_ARG, "b200_unletterbox_boxes: null argument");
  UlbParams p;
  p.pad_top = (float)padding[0]; p.pad_bottom = (float)padding[1]; p.pad_left = (float)padding[2]; p.pad_right = (float)padding[3];
  p.old_w = (float)image_size_old[0]; p.old_h = (float)image_size_old[1];
  p.geometry = nullptr;
  return ulb_launch("b200_unletterbox_boxes", p, boxes, counts, B, max_rows, image_size, out_boxes, out_index, out_count, stream);
}

extern "C" int b200_unletterbox_boxes_batch(const float* boxes, const int32_t* counts, int B, int max_rows,
                                            const int32_t image_size[2], const int32_t* geometry, int32_t* out_boxes,
                                            int32_t* out_index, int32_t* out_count, void* stream) {
  B200_REQUIRE(B <= 0 || geometry, B200_ERR_BAD_ARG, "b200_unletterbox_boxes_batch: null geometry");
  UlbParams p;
  p.pad_top = p.pad_bottom = p.pad_left = p.pad_right = p.old_w = p.old_h = 0.0f;
  p.geometry = geometry;
  return ulb_launch("b200_unletterbox_boxes_batch", p, boxes, counts, B, max_rows, image_size, out_boxes, out_index, out_count,
                    stream);
}
