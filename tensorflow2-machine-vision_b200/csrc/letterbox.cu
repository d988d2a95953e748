// letterbox.cu — the image pre-processing of the serving path (SURVEY §8f N4): ImageHelper.opencvProportionalResize
// (utils/image_helper.py:293-325, constant border) and the colour swap / float conversion that `predict` applies to
// its result (views/object_detection.py:50-62), in one launch.
//
// The resize is cv2.resize(..., interpolation=cv2.INTER_AREA) of an 8-bit 3-channel image.  OpenCV's arithmetic is
// reproduced bit for bit.  When the image shrinks (or keeps its size) in both directions — the serving case — it is a
// true area resize:
//   * both scale factors integral: int32 block sum, saturate_cast<uchar>(sum * (1.f / area)) (round half to even); the
//     2x2 block has its own form, (a + b + c + d + 2) >> 2;
//   * otherwise: per destination index a run of source taps — an optional partial tap, full taps of weight 1/cell, an
//     optional partial tap — whose fp32 weights come from fp64 interval arithmetic; a horizontal pass accumulates
//     S * alpha in fp32 in tap order, the vertical pass accumulates beta * row the same way, one rounding at the end.
// When it grows in either direction OpenCV does not do an area resize at all: INTER_AREA falls back to its 8-bit
// bilinear with "area mode" coefficients — left neighbour floor(d * scale), weight fx = (d+1) - (s+1) * inv_scale kept
// to its fractional part, both weights rounded to 11-bit fixed point; the horizontal pass is S0*a0 + S1*a1 in int32 and
// the vertical pass (((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2.
// Every destination pixel is independent, so a thread recomputes its own taps (a few fp64 operations) instead of
// reading tables: no host-side table build, no upload, one kernel.
//
// Output: the letterboxed uint8 image in the input's channel order (what opencvProportionalResize returns) and / or
// the float32 network input with the channels reversed and divided by 255 (predict's cvtColor + astype + / 255).
#include "detmath.h"
#include "common.cuh"

#include <cstdio>
#include <cstring>
#include <vector>

enum { LB_GENERIC = 0, LB_BLOCK = 1, LB_BLOCK_2X2 = 2, LB_LINEAR = 3 };

// One frame of a launch.  The fp64 scales are not stored: the kernel recomputes them from rw / sw and rh / sh with the
// same correctly rounded operations the host uses to pick the mode, so 48 bytes per frame fit LB_MAX_IMAGES frames in
// the classic 4 KB kernel-argument block (no workspace, no upload: a batch stays capturable in a CUDA graph).
struct LbImage {
  const uint8_t* img;  // [sh, sw, 3]
  int sh, sw, rw, rh, top, left;
  int mode, isx, isy;
};

#define LB_MAX_IMAGES 84  // frames per launch; a longer batch is split into several launches

struct LbBatch {
  uint8_t* out_u8;     // optional [n, out_h, out_w, 3]
  float* out_f32;      // optional [n, out_h, out_w, 3], channels reversed, / 255
  int32_t* geometry;   // optional [n, 6] top, bottom, left, right, sw, sh (what b200_unletterbox_boxes_batch reads)
  int out_w, out_h, bg0, bg1, bg2;
  LbImage im[LB_MAX_IMAGES];
};
static_assert(sizeof(LbBatch) <= 4096, "LbBatch must fit the 4 KB kernel-argument block");

struct LbAxis {
  int sx1, sx2;             // full taps sx1 .. sx2-1
  bool has_first, has_last; // partial taps at sx1-1 and sx2
  float a_first, a_mid, a_last;
};

// computeResizeAreaTab for one destination index (fp64, every operation rounded separately)
__device__ __forceinline__ LbAxis lb_axis(int d, int ssize, double scale) {
  LbAxis t;
  const double f1 = __dmul_rn((double)d, scale), f2 = __dadd_rn(f1, scale);
  const double cell = fmin(scale, __dsub_rn((double)ssize, f1));
  int sx1 = (int)ceil(f1), sx2 = (int)floor(f2);
  sx2 = min(sx2, ssize - 1);
  sx1 = min(sx1, sx2);
  const double dl = __dsub_rn((double)sx1, f1), dr = __dsub_rn(f2, (double)sx2);
  t.sx1 = sx1; t.sx2 = sx2;
  t.has_first = dl > 1e-3;
  t.has_last = dr > 1e-3;
  t.a_first = (float)__ddiv_rn(dl, cell);
  t.a_mid = (float)__ddiv_rn(1.0, cell);
  t.a_last = (float)__ddiv_rn(fmin(fmin(dr, 1.0), cell), cell);
  return t;
}

__device__ __forceinline__ int lb_saturate(int v) { return min(max(v, 0), 255); }

// one axis of the bilinear fallback: left source index and the two fixed-point weights (INTER_RESIZE_COEF_BITS = 11)
__device__ __forceinline__ void lb_linear(int d, int ssize, double inv, double scale, int& s, int& w0, int& w1) {
  s = (int)floor(__dmul_rn((double)d, scale));
  float f = (float)__dsub_rn((double)(d + 1), __dmul_rn((double)(s + 1), inv));
  f = (f <= 0.0f) ? 0.0f : DM_SUB(f, floorf(f));
  if (s < 0) { f = 0.0f; s = 0; }
  if (s >= ssize - 1) { f = 0.0f; s = ssize - 1; }
  w0 = min(max(__float2int_rn(DM_MUL(DM_SUB(1.0f, f), 2048.0f)), -32768), 32767);  // saturate_cast<short>
  w1 = min(max(__float2int_rn(DM_MUL(f, 2048.0f)), -32768), 32767);
}

// grid (out_w / 32, out_h / 8, frames of this launch); blockIdx.z selects the frame
__global__ void __launch_bounds__(256) letterbox_kernel(const __grid_constant__ LbBatch b) {
  const LbImage& p = b.im[blockIdx.z];
  const size_t plane = (size_t)b.out_h * b.out_w * 3;
  if (b.geometry && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x < 6) {
    const int t = (int)threadIdx.x;
    const int g = t == 0 ? p.top : t == 1 ? b.out_h - p.rh - p.top : t == 2 ? p.left : t == 3 ? b.out_w - p.rw - p.left : t == 4 ? p.sw : p.sh;
    b.geometry[(size_t)blockIdx.z * 6 + t] = g;
  }
  const int ox = blockIdx.x * 32 + (int)(threadIdx.x & 31), oy = blockIdx.y * 8 + (int)(threadIdx.x >> 5);
  if (ox >= b.out_w || oy >= b.out_h) return;
  const int dx = ox - p.left, dy = oy - p.top;
  int v0 = b.bg0, v1 = b.bg1, v2 = b.bg2;  // copyMakeBorder(BORDER_CONSTANT)
  if (dx >= 0 && dx < p.rw && dy >= 0 && dy < p.rh) {
    // cv::resize: inv_scale = dsize / ssize, scale = 1 / inv_scale (the host computes the same to choose the mode)
    const double inv_x = __ddiv_rn((double)p.rw, (double)p.sw), inv_y = __ddiv_rn((double)p.rh, (double)p.sh);
    const double scale_x = __ddiv_rn(1.0, inv_x), scale_y = __ddiv_rn(1.0, inv_y);
    if (p.mode == LB_GENERIC) {
      const LbAxis ax = lb_axis(dx, p.sw, scale_x), ay = lb_axis(dy, p.sh, scale_y);
      float s0 = 0.f, s1 = 0.f, s2 = 0.f;
      // source rows in tap order: first partial, full rows, last partial
      const int y_begin = ay.has_first ? ay.sx1 - 1 : ay.sx1, y_end = ay.has_last ? ay.sx2 + 1 : ay.sx2;
      for (int sy = y_begin; sy < y_end; ++sy) {
        const float beta = (sy < ay.sx1) ? ay.a_first : ((sy < ay.sx2) ? ay.a_mid : ay.a_last);
        const uint8_t* S = p.img + (size_t)max(sy, 0) * p.sw * 3;
        float b0 = 0.f, b1 = 0.f, b2 = 0.f;
        if (ax.has_first) {
          const uint8_t* q = S + (size_t)max(ax.sx1 - 1, 0) * 3;
          b0 = DM_ADD(b0, DM_MUL((float)__ldg(q), ax.a_first));
          b1 = DM_ADD(b1, DM_MUL((float)__ldg(q + 1), ax.a_first));
          b2 = DM_ADD(b2, DM_MUL((float)__ldg(q + 2), ax.a_first));
        }
        for (int sx = ax.sx1; sx < ax.sx2; ++sx) {
          const uint8_t* q = S + (size_t)sx * 3;
          b0 = DM_ADD(b0, DM_MUL((float)__ldg(q), ax.a_mid));
          b1 = DM_ADD(b1, DM_MUL((float)__ldg(q + 1), ax.a_mid));
          b2 = DM_ADD(b2, DM_MUL((float)__ldg(q + 2), ax.a_mid));
        }
        if (ax.has_last) {
          const uint8_t* q = S + (size_t)ax.sx2 * 3;
          b0 = DM_ADD(b0, DM_MUL((float)__ldg(q), ax.a_last));
          b1 = DM_ADD(b1, DM_MUL((float)__ldg(q + 1), ax.a_last));
          b2 = DM_ADD(b2, DM_MUL((float)__ldg(q + 2), ax.a_last));
        }
        s0 = DM_ADD(s0, DM_MUL(beta, b0));
        s1 = DM_ADD(s1, DM_MUL(beta, b1));
        s2 = DM_ADD(s2, DM_MUL(beta, b2));
      }
      v0 = lb_saturate(__float2int_rn(s0)); v1 = lb_saturate(__float2int_rn(s1)); v2 = lb_saturate(__float2int_rn(s2));
    } else if (p.mode == LB_LINEAR) {
      int sx, a0, a1, sy, b0, b1;
      lb_linear(dx, p.sw, inv_x, scale_x, sx, a0, a1);
      lb_linear(dy, p.sh, inv_y, scale_y, sy, b0, b1);
      const int sx1 = min(sx + 1, p.sw - 1);
      const uint8_t* R0 = p.img + (size_t)min(max(sy, 0), p.sh - 1) * p.sw * 3;
      const uint8_t* R1 = p.img + (size_t)min(max(sy + 1, 0), p.sh - 1) * p.sw * 3;
      int v[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const int h0 = (int)__ldg(R0 + sx * 3 + c) * a0 + (int)__ldg(R0 + sx1 * 3 + c) * a1;
        const int h1 = (int)__ldg(R1 + sx * 3 + c) * a0 + (int)__ldg(R1 + sx1 * 3 + c) * a1;
        v[c] = ((((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2) & 0xff;  // uchar(...) truncates
      }
      v0 = v[0]; v1 = v[1]; v2 = v[2];
    } else {
      int s0 = 0, s1 = 0, s2 = 0;
      for (int ky = 0; ky < p.isy; ++ky) {
        const uint8_t* S = p.img + ((size_t)(dy * p.isy + ky) * p.sw + (size_t)dx * p.isx) * 3;
        for (int kx = 0; kx < p.isx; ++kx) {
          s0 += __ldg(S + kx * 3); s1 += __ldg(S + kx * 3 + 1); s2 += __ldg(S + kx * 3 + 2);
        }
      }
      if (p.mode == LB_BLOCK_2X2) {
        v0 = (s0 + 2) >> 2; v1 = (s1 + 2) >> 2; v2 = (s2 + 2) >> 2;
      } else {
        const float inv_area = __fdiv_rn(1.0f, (float)(p.isx * p.isy));
        v0 = lb_saturate(__float2int_rn(DM_MUL((float)s0, inv_area)));
        v1 = lb_saturate(__float2int_rn(DM_MUL((float)s1, inv_area)));
        v2 = lb_saturate(__float2int_rn(DM_MUL((float)s2, inv_area)));
      }
    }
  }
  const size_t o = plane * blockIdx.z + ((size_t)oy * b.out_w + ox) * 3;
  if (b.out_u8) { b.out_u8[o] = (uint8_t)v0; b.out_u8[o + 1] = (uint8_t)v1; b.out_u8[o + 2] = (uint8_t)v2; }
  if (b.out_f32) {  // cvtColor(BGR2RGB), astype(float32), / 255
    b.out_f32[o] = DM_DIV((float)v2, 255.0f); b.out_f32[o + 1] = DM_DIV((float)v1, 255.0f); b.out_f32[o + 2] = DM_DIV((float)v0, 255.0f);
  }
}

// Validates one frame and plans it: the proportional size of image_helper.py:297-303, the border and OpenCV's
// INTER_AREA mode.  Errors name the frame when `index` >= 0 (a batch).
static int lb_plan(const char* who, int index, const uint8_t* img, int height, int width, int channels, int out_width,
                   int out_height, LbImage* im, int32_t padding_out[4], int32_t* resized_wh_out) {
  char at[96];
  if (index >= 0) snprintf(at, sizeof(at), "%s: image %d", who, index); else snprintf(at, sizeof(at), "%s", who);
  B200_REQUIRE(img, B200_ERR_BAD_ARG, "%s: null image pointer", at);
  B200_REQUIRE(height > 0 && width > 0 && out_width > 0 && out_height > 0, B200_ERR_BAD_ARG, "%s: bad sizes", at);
  B200_REQUIRE(height < (1 << 24) && width < (1 << 24) && out_width < (1 << 16) && out_height < (1 << 16), B200_ERR_BAD_ARG,
               "%s: image too large", at);
  B200_REQUIRE(channels == 3, B200_ERR_UNSUPPORTED, "%s: 3-channel 8-bit images only (got %d channels)", at, channels);
  // image_helper.py:297-303 in Python float (= C double) arithmetic; int() truncates
  int rw, rh;
  if ((double)width / (double)height > (double)out_width / (double)out_height) {
    rw = out_width;
    rh = (int)(((double)height / (double)width) * (double)rw);
  } else {
    rh = out_height;
    rw = (int)(((double)width / (double)height) * (double)rh);
  }
  B200_REQUIRE(rw >= 1 && rh >= 1, B200_ERR_BAD_ARG, "%s: the resized image would be empty (%d x %d), as cv2.resize fails", at, rw, rh);
  const double scale_x = 1.0 / ((double)rw / (double)width), scale_y = 1.0 / ((double)rh / (double)height);
  const bool area = scale_x >= 1.0 && scale_y >= 1.0;  // otherwise INTER_AREA is OpenCV's bilinear fallback
  const int isx = (int)nearbyint(scale_x), isy = (int)nearbyint(scale_y);
  const bool blocky = fabs(scale_x - isx) < 2.220446049250313e-16 && fabs(scale_y - isy) < 2.220446049250313e-16;
  im->img = img; im->sh = height; im->sw = width; im->rw = rw; im->rh = rh;
  im->top = (out_height - rh) / 2;
  im->left = (out_width - rw) / 2;
  im->mode = !area ? LB_LINEAR : (!blocky ? LB_GENERIC : ((isx == 2 && isy == 2) ? LB_BLOCK_2X2 : LB_BLOCK));
  im->isx = isx; im->isy = isy;
  padding_out[0] = im->top; padding_out[1] = out_height - rh - im->top;
  padding_out[2] = im->left; padding_out[3] = out_width - rw - im->left;
  if (resized_wh_out) { resized_wh_out[0] = rw; resized_wh_out[1] = rh; }
  return B200_OK;
}

// Launches planned frames, LB_MAX_IMAGES per launch.
static int lb_launch(int N, const LbImage* ims, int out_width, int out_height, const uint8_t bg_color[3], uint8_t* out_u8,
                     float* out_f32, int32_t* geometry_out, cudaStream_t stream) {
  const size_t plane = (size_t)out_height * out_width * 3;
  for (int c0 = 0; c0 < N; c0 += LB_MAX_IMAGES) {
    const int n = min(N - c0, LB_MAX_IMAGES);
    LbBatch b;
    b.out_u8 = out_u8 ? out_u8 + plane * c0 : nullptr;
    b.out_f32 = out_f32 ? out_f32 + plane * c0 : nullptr;
    b.geometry = geometry_out ? geometry_out + (size_t)6 * c0 : nullptr;
    b.out_w = out_width; b.out_h = out_height;
    b.bg0 = bg_color[0]; b.bg1 = bg_color[1]; b.bg2 = bg_color[2];
    memcpy(b.im, ims + c0, sizeof(LbImage) * n);
    const dim3 grid((out_width + 31) / 32, (out_height + 7) / 8, n);
    letterbox_kernel<<<grid, 256, 0, stream>>>(b);
    B200_LAUNCH_CHECK();
  }
  return B200_OK;
}

extern "C" int b200_letterbox_image(const uint8_t* img, int height, int width, int channels, int out_width, int out_height,
                                    const uint8_t bg_color[3], uint8_t* out_u8, float* out_f32, int32_t padding_out[4],
                                    int32_t resized_wh_out[2], void* stream) {
  B200_REQUIRE(img && bg_color && padding_out, B200_ERR_BAD_ARG, "b200_letterbox_image: null argument");
  B200_REQUIRE(out_u8 || out_f32, B200_ERR_BAD_ARG, "b200_letterbox_image: no output buffer");
  LbImage im;
  const int st = lb_plan("b200_letterbox_image", -1, img, height, width, channels, out_width, out_height, &im, padding_out,
                         resized_wh_out);
  if (st != B200_OK) return st;
  return lb_launch(1, &im, out_width, out_height, bg_color, out_u8, out_f32, nullptr, (cudaStream_t)stream);
}

extern "C" int b200_letterbox_batch(int N, const uint8_t* const imgs[], const int32_t* hw, int channels, int out_width,
                                    int out_height, const uint8_t bg_color[3], uint8_t* out_u8, float* out_f32,
                                    int32_t* padding_out, int32_t* resized_wh_out, int32_t* geometry_out, void* stream) {
  B200_REQUIRE(N >= 0, B200_ERR_BAD_ARG, "b200_letterbox_batch: bad image count %d", N);
  if (N == 0) return B200_OK;
  B200_REQUIRE(imgs && hw && bg_color && padding_out, B200_ERR_BAD_ARG, "b200_letterbox_batch: null argument");
  B200_REQUIRE(out_u8 || out_f32, B200_ERR_BAD_ARG, "b200_letterbox_batch: no output buffer");
  std::vector<LbImage> ims((size_t)N);
  for (int i = 0; i < N; ++i) {  // every frame is checked before anything is launched
    const int st = lb_plan("b200_letterbox_batch", i, imgs[i], hw[2 * i], hw[2 * i + 1], channels, out_width, out_height, &ims[i],
                           padding_out + 4 * i, resized_wh_out ? resized_wh_out + 2 * i : nullptr);
    if (st != B200_OK) return st;
  }
  return lb_launch(N, ims.data(), out_width, out_height, bg_color, out_u8, out_f32, geometry_out, (cudaStream_t)stream);
}
