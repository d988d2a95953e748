// effdet_loss.cu — EfficientDet training loss: FocalLoss (losses/focal_loss.py:26-52) + Keras mean reduction,
// BoxLoss / Huber(delta=0.1) (losses/box_loss.py:17-29) and the aggregation of
// EfficientDetNetTrain._get_loss (efficientnet/efficientdet_net_train.py:41-52), L2-regularisation excluded
// (it is over model weights and stays in the TF graph).
//
//   K8a focal_box_partials_kernel  one pass over every level: class logits + one-hot targets as 128-bit streaming
//        loads (the HBM-bound part: 2 x 15.9 MB per D0 image), box outputs/targets/masks per anchor; per-CTA fp64
//        partial sums of {focal_l, huber_l, positives}.  Element math uses MUFU exp/log/rcp/sqrt: the loss is a
//        continuous output with a 1e-4 relative budget; nothing discrete depends on it.
//   K8b focal_box_reduce_kernel    fixed-order reduction of the partials -> sums[2L+1] (fp64, un-normalised) so a
//        data-parallel caller can all-reduce them before normalising.
//   K8c focal_box_finalize_kernel  num_pos = sum(mask)+1; box_l = huber_l/(4 num_pos); focal_l = focal_l/num_pos/numel_l
//        (FocalLoss.call divides per element, Keras SUM_OVER_BATCH_SIZE then takes the mean over the level, Q14);
//        loss = sum_l (50 box_l + focal_l) in fp32 in the reference's order.
#include "common.cuh"
#include "detmath.h"
#include "exchange.cuh"
#include "effdet_focal.cuh"
#include "effdet_anchor.cuh"

#define EL_MAX_LEVELS 8
#define EL_THREADS 256

struct ElParams {
  int num_levels;
  const float4* cls_pred[EL_MAX_LEVELS];
  const float4* cls_true[EL_MAX_LEVELS];
  const int32_t* cls_index[EL_MAX_LEVELS];     // sparse-target mode: class id per anchor instead of the one-hot tensor
  int C;
  unsigned long long cls_vec[EL_MAX_LEVELS];   // float4 count of the class tensors
  const float* cls_pred_tail[EL_MAX_LEVELS]; const float* cls_true_tail[EL_MAX_LEVELS]; int cls_tail[EL_MAX_LEVELS];
  const float4* box_pred[EL_MAX_LEVELS];
  const float4* box_true[EL_MAX_LEVELS];
  const unsigned char* mask[EL_MAX_LEVELS];
  unsigned long long anchors[EL_MAX_LEVELS];   // B*H*W*A
  int cta_base[EL_MAX_LEVELS + 1];
  float alpha, gamma, delta, label_smoothing;
  double* partials;  // [n_cta, 3]
};

// G15: gamma == 1.5 (the reference's value, global_params.py:186) — q^1.5 = q*sqrt(q) without a per-element branch
template <bool G15>
__global__ void __launch_bounds__(EL_THREADS) focal_box_partials_kernel(ElParams p) {
  __shared__ double s_red[EL_THREADS / 32][3];
  int l = 0;
#pragma unroll
  for (int k = 1; k < EL_MAX_LEVELS; ++k) if (k < p.num_levels && (int)blockIdx.x >= p.cta_base[k]) l = k;
  const int ncta = p.cta_base[l + 1] - p.cta_base[l];
  const int cta = blockIdx.x - p.cta_base[l];
  const unsigned long long stride = (unsigned long long)ncta * EL_THREADS;
  float f0 = 0.f, f1 = 0.f;  // two fp32 accumulators per thread, folded into fp64 per thread at the end
  double focal = 0.0;
  const float4* __restrict__ cp = p.cls_pred[l];
  const float4* __restrict__ ct = p.cls_true[l];
  const unsigned long long nv = p.cls_vec[l];
  unsigned long long i = (unsigned long long)cta * EL_THREADS + threadIdx.x;
  int it = 0;
  const int32_t* __restrict__ ci = p.cls_index[l];
  if (ci) {
    // sparse-target mode: sum over every logit of the background term, then per anchor swap the term of its class
    // for the y = 1 one
    const float oma = 1.0f - p.alpha, hls = 0.5f * p.label_smoothing;
#pragma unroll 2
    for (; i < nv; i += stride) {
      const float4 x = __ldcs(cp + i);
      f0 += el_focal_bg<G15>(x.x, oma, p.gamma, hls) + el_focal_bg<G15>(x.y, oma, p.gamma, hls);
      f1 += el_focal_bg<G15>(x.z, oma, p.gamma, hls) + el_focal_bg<G15>(x.w, oma, p.gamma, hls);
      if ((++it & 63) == 0) { focal += (double)f0 + (double)f1; f0 = f1 = 0.f; }
    }
    if (cta == 0 && (int)threadIdx.x < p.cls_tail[l]) f0 += el_focal_bg<G15>(p.cls_pred_tail[l][threadIdx.x], oma, p.gamma, hls);
    const float* __restrict__ logits = reinterpret_cast<const float*>(cp);
    const unsigned long long n_anchor = (nv * 4ull + (unsigned long long)p.cls_tail[l]) / (unsigned long long)p.C;
    for (unsigned long long a = (unsigned long long)cta * EL_THREADS + threadIdx.x; a < n_anchor; a += stride) {
      const int cls = __ldg(ci + a);
      if (cls >= 0 && cls < p.C) {  // tf.one_hot: ids outside [0, C) give an all-zero row
        const float x = __ldg(logits + a * (unsigned long long)p.C + cls);
        f0 += el_focal<G15>(1.0f, x, p.alpha, p.gamma, p.label_smoothing) - el_focal_bg<G15>(x, oma, p.gamma, hls);
      }
    }
  } else {
#pragma unroll 2
    for (; i < nv; i += stride) {
      const float4 x = __ldcs(cp + i);
      const float4 y = __ldcs(ct + i);
      f0 += el_focal<G15>(y.x, x.x, p.alpha, p.gamma, p.label_smoothing) + el_focal<G15>(y.y, x.y, p.alpha, p.gamma, p.label_smoothing);
      f1 += el_focal<G15>(y.z, x.z, p.alpha, p.gamma, p.label_smoothing) + el_focal<G15>(y.w, x.w, p.alpha, p.gamma, p.label_smoothing);
      if ((++it & 63) == 0) { focal += (double)f0 + (double)f1; f0 = f1 = 0.f; }
    }
    if (cta == 0 && (int)threadIdx.x < p.cls_tail[l])
      f0 += el_focal<G15>(p.cls_true_tail[l][threadIdx.x], p.cls_pred_tail[l][threadIdx.x], p.alpha, p.gamma, p.label_smoothing);
  }
  focal += (double)f0 + (double)f1;
  float hub = 0.f;
  unsigned int pos = 0;
  const unsigned long long na = p.anchors[l];
  for (unsigned long long a = (unsigned long long)cta * EL_THREADS + threadIdx.x; a < na; a += stride) {
    const float4 o = __ldcs(p.box_pred[l] + a);
    const float4 t = __ldcs(p.box_true[l] + a);
    hub += el_huber(t.x, o.x, p.delta) + el_huber(t.y, o.y, p.delta) + el_huber(t.z, o.z, p.delta) + el_huber(t.w, o.w, p.delta);
    pos += p.mask[l][a] ? 1u : 0u;
  }
  double v0 = warp_sum_d(focal), v1 = warp_sum_d((double)hub), v2 = warp_sum_d((double)pos);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { s_red[warp][0] = v0; s_red[warp][1] = v1; s_red[warp][2] = v2; }
  __syncthreads();
  if (threadIdx.x < 3) {
    double s = 0.0;
    for (int w = 0; w < EL_THREADS / 32; ++w) s += s_red[w][threadIdx.x];
    p.partials[(size_t)blockIdx.x * 3 + threadIdx.x] = s;
  }
}

struct ElReduce { const double* partials; int num_levels; int cta_base[EL_MAX_LEVELS + 1]; double* sums; };

// sums layout: [0..L) focal_l, [L..2L) huber_l, [2L] positives
__global__ void __launch_bounds__(256) focal_box_reduce_kernel(ElReduce r) {
  __shared__ double s_red[8][3];
  const int l = blockIdx.x;
  double a[3] = {0.0, 0.0, 0.0};
  for (int c = r.cta_base[l] + threadIdx.x; c < r.cta_base[l + 1]; c += 256) {
    a[0] += r.partials[(size_t)c * 3 + 0]; a[1] += r.partials[(size_t)c * 3 + 1]; a[2] += r.partials[(size_t)c * 3 + 2];
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 3; ++k) { const double v = warp_sum_d(a[k]); if (lane == 0) s_red[warp][k] = v; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double s[3] = {0.0, 0.0, 0.0};
    for (int w = 0; w < 8; ++w) for (int k = 0; k < 3; ++k) s[k] += s_red[w][k];
    r.sums[l] = s[0];
    r.sums[r.num_levels + l] = s[1];
    atomicAdd(&r.sums[2 * r.num_levels], s[2]);  // integer-valued: exact and order-independent
  }
}

struct ElFinalize {
  double* sums; int num_levels; double numel[EL_MAX_LEVELS]; float* parts; float* loss; float* num_pos;
  B200Exchange xchg;  // data parallel: the 2L+1 sums are added over the ranks here first (world 1: no-op)
};

__global__ void __launch_bounds__(32) focal_box_finalize_kernel(ElFinalize f) {
  const int L = f.num_levels;
  if (f.xchg.world > 1) {
    // num_positives is a batch-wide count (edt:43-46): the un-normalised sums of every rank are added (fp64, rank order)
    // before anything is divided; the global sums are written back for the backward pass
    const int lane = threadIdx.x, n = 2 * L + 1;
    double v = lane < n ? f.sums[lane] : 0.0;
    v = xchg_allreduce_warp<double>(f.xchg, v, n);
    if (lane < n) f.sums[lane] = v;
    __syncwarp();
  }
  if (threadIdx.x != 0) return;
  const float npos = DM_ADD((float)f.sums[2 * L], 1.0f);         // edt:43-46
  if (f.num_pos) *f.num_pos = npos;
  float loss = 0.0f;
  for (int l = 0; l < L; ++l) {
    const float box = DM_DIV((float)f.sums[L + l], DM_MUL(npos, 4.0f));            // box_loss.py:23,29
    const float focal = (float)((f.sums[l] / (double)npos) / f.numel[l]);          // focal_loss.py:52 + Keras mean
    if (f.parts) { f.parts[2 * l] = box; f.parts[2 * l + 1] = focal; }
    loss = DM_ADD(loss, DM_ADD(DM_MUL(box, 50.0f), focal));                         // edt:51
  }
  *f.loss = loss;
}

// ---- backward (SURVEY §8f N1): d _get_loss / d class logits and d / d box outputs --------------------------
// focal: f = af*mod*ce, mod = q^gamma, q = 1-p_t, p_t = y p + (1-y)(1-p):
//   df/dx = af * ( gamma q^(gamma-1) * (-(2y-1) p (1-p)) * ce + mod * (p - y_smoothed) );  scaled by 1/(num_pos*numel_l)
// box:   d huber/d o = (|e| <= delta ? e : delta sign(e)) for target != 0, scaled by 50/(4 num_pos)
// num_pos comes from the (all-reduced) partial sums and is a constant of the targets.
struct ElGradParams {
  int num_levels;
  const float4* cls_pred[EL_MAX_LEVELS]; const float4* cls_true[EL_MAX_LEVELS]; float4* cls_grad[EL_MAX_LEVELS];
  const int32_t* cls_index[EL_MAX_LEVELS];  // sparse-target mode: class id per anchor instead of cls_true
  int C;
  unsigned long long cls_vec[EL_MAX_LEVELS];
  int cls_tail[EL_MAX_LEVELS];  // floats after the last whole float4
  const float4* box_pred[EL_MAX_LEVELS]; const float4* box_true[EL_MAX_LEVELS]; float4* box_grad[EL_MAX_LEVELS];
  unsigned long long anchors[EL_MAX_LEVELS];
  double numel[EL_MAX_LEVELS];
  int cta_base[EL_MAX_LEVELS + 1];
  float alpha, gamma, delta, label_smoothing;
  const double* sums;  // [2L+1], sums[2L] = positives
};

// The focal derivative and, from the same intermediates, the focal value af*mod*ce (4 MUFU operations for both).
__device__ __forceinline__ float el_focal_value_grad(float y, float x, float alpha, float gamma, float ls, float& value) {
  const float e = el_ex2(-1.4426950408889634f * fabsf(x));
  const float r = el_rcp(1.0f + e);
  const float p = (x >= 0.0f) ? r : e * r;
  const float p_t = y * p + (1.0f - y) * (1.0f - p);
  const float af = y * alpha + (1.0f - y) * (1.0f - alpha);
  const float q = fmaxf(1.0f - p_t, 0.0f);
  const float sq = el_sqrt(q);
  const float mod = (gamma == 1.5f) ? q * sq : __powf(q, gamma);
  const float dmod = (gamma == 1.5f) ? 1.5f * sq : (q > 0.0f ? gamma * __powf(q, gamma - 1.0f) : 0.0f);
  const float ys = y * (1.0f - ls) + 0.5f * ls;
  const float ce = fmaxf(x, 0.0f) - x * ys - 0.6931471805599453f * el_lg2(r);
  const float dq = -(2.0f * y - 1.0f) * p * (1.0f - p);
  value = af * mod * ce;
  return af * (dmod * dq * ce + mod * (p - ys));
}

__device__ __forceinline__ float el_focal_grad(float y, float x, float alpha, float gamma, float ls) {
  float unused;
  return el_focal_value_grad(y, x, alpha, gamma, ls, unused);
}

__device__ __forceinline__ float el_huber_grad(float t, float o, float delta) {
  if (t == 0.0f) return 0.0f;
  const float e = o - t;
  return fabsf(e) <= delta ? e : copysignf(delta, e);
}

__global__ void __launch_bounds__(EL_THREADS) focal_box_grad_kernel(ElGradParams p) {
  int l = 0;
#pragma unroll
  for (int k = 1; k < EL_MAX_LEVELS; ++k) if (k < p.num_levels && (int)blockIdx.x >= p.cta_base[k]) l = k;
  const int ncta = p.cta_base[l + 1] - p.cta_base[l];
  const int cta = blockIdx.x - p.cta_base[l];
  const unsigned long long stride = (unsigned long long)ncta * EL_THREADS;
  const float npos = (float)p.sums[2 * p.num_levels] + 1.0f;
  const float cs = (float)(1.0 / ((double)npos * p.numel[l]));
  const float bs = 50.0f / (4.0f * npos);
  if (p.cls_grad[l]) {
    const unsigned long long nv = p.cls_vec[l];
    const int32_t* __restrict__ ci = p.cls_index[l];
#pragma unroll 2
    for (unsigned long long i = (unsigned long long)cta * EL_THREADS + threadIdx.x; i < nv; i += stride) {
      const float4 x = __ldcs(p.cls_pred[l] + i);
      float4 y;
      if (ci) {
        // the one-hot row generate_targets would have written: 1 at the anchor's class id, ids outside [0, C) -> zeros
        const unsigned long long e = i * 4ull, a0 = e / (unsigned long long)p.C;
        const int c0 = (int)(e - a0 * (unsigned long long)p.C);
        const int id0 = __ldg(ci + a0);
        const int id1 = (c0 + 3 >= p.C) ? __ldg(ci + a0 + 1) : 0;  // a float4 may straddle two anchors (C >= 4 here)
        float yy[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int c = c0 + k;
          yy[k] = (c < p.C) ? ((c == id0) ? 1.0f : 0.0f) : ((c - p.C == id1) ? 1.0f : 0.0f);
        }
        y = make_float4(yy[0], yy[1], yy[2], yy[3]);
      } else {
        y = __ldcs(p.cls_true[l] + i);
      }
      float4 g;
      g.x = cs * el_focal_grad(y.x, x.x, p.alpha, p.gamma, p.label_smoothing);
      g.y = cs * el_focal_grad(y.y, x.y, p.alpha, p.gamma, p.label_smoothing);
      g.z = cs * el_focal_grad(y.z, x.z, p.alpha, p.gamma, p.label_smoothing);
      g.w = cs * el_focal_grad(y.w, x.w, p.alpha, p.gamma, p.label_smoothing);
      __stcs(p.cls_grad[l] + i, g);
    }
    if (cta == 0 && (int)threadIdx.x < p.cls_tail[l]) {
      const unsigned long long e = nv * 4ull + threadIdx.x;
      float yt;
      if (p.cls_index[l]) {
        const unsigned long long a = e / (unsigned long long)p.C;
        yt = ((int)(e - a * (unsigned long long)p.C) == __ldg(p.cls_index[l] + a)) ? 1.0f : 0.0f;
      } else {
        yt = reinterpret_cast<const float*>(p.cls_true[l])[e];
      }
      reinterpret_cast<float*>(p.cls_grad[l])[e] =
          cs * el_focal_grad(yt, reinterpret_cast<const float*>(p.cls_pred[l])[e], p.alpha, p.gamma, p.label_smoothing);
    }
  }
  if (p.box_grad[l]) {
    const unsigned long long na = p.anchors[l];
    for (unsigned long long a = (unsigned long long)cta * EL_THREADS + threadIdx.x; a < na; a += stride) {
      const float4 o = __ldcs(p.box_pred[l] + a);
      const float4 t = __ldcs(p.box_true[l] + a);
      __stcs(p.box_grad[l] + a, make_float4(bs * el_huber_grad(t.x, o.x, p.delta), bs * el_huber_grad(t.y, o.y, p.delta),
                                             bs * el_huber_grad(t.z, o.z, p.delta), bs * el_huber_grad(t.w, o.w, p.delta)));
    }
  }
}

// ---- host side ------------------------------------------------------------------------------------
// CTAs proportional to the class-tensor size of each level, `budget` in total (at most budget + num_levels after
// rounding up), at least 1 per level.
static int el_cta_plan_budget(int num_levels, const unsigned long long* cls_elems, int* cta_base, int budget) {
  unsigned long long tot = 0;
  for (int l = 0; l < num_levels; ++l) tot += cls_elems[l];
  int c = 0;
  for (int l = 0; l < num_levels; ++l) {
    cta_base[l] = c;
    unsigned long long want = tot ? (cls_elems[l] * (unsigned long long)budget + tot - 1) / tot : 1;
    const unsigned long long max_useful = (cls_elems[l] / 4 + EL_THREADS - 1) / EL_THREADS;
    if (want > max_useful) want = max_useful;
    if (want < 1) want = 1;
    c += (int)want;
  }
  for (int l = num_levels; l <= EL_MAX_LEVELS; ++l) cta_base[l] = c;
  return c;
}

static int el_cta_plan(int num_levels, const unsigned long long* cls_elems, int* cta_base) {
  // ~64 CTAs per SM.  Measured on D0 B=128: 8 per SM 0.80 ms, 16 0.75, 32 0.71, 64 0.69 (92 % of the copy bandwidth),
  // 96 0.69 — many short CTAs keep the tail of every level busy.
  return el_cta_plan_budget(num_levels, cls_elems, cta_base, b200_sm_count() * 64);
}

// FocalLoss.call (focal_loss.py:26-52): the per-element tensor alpha*mod*ce/normalizer.
__global__ void focal_elementwise_kernel(const float* __restrict__ y, const float* __restrict__ x, size_t n, float normalizer,
                                         float alpha, float gamma, float ls, float* __restrict__ out) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[i] = el_focal(y[i], x[i], alpha, gamma, ls) / normalizer;
}

extern "C" int b200_focal_elementwise(const float* y_true, const float* y_pred, size_t n, float normalizer, float alpha,
                                      float gamma, float label_smoothing, float* out, void* stream) {
  if (n == 0) return B200_OK;
  B200_REQUIRE(y_true && y_pred && out, B200_ERR_BAD_ARG, "b200_focal_elementwise: null pointer");
  size_t blocks = (n + 255) / 256;
  const size_t cap = (size_t)b200_sm_count() * 16;
  if (blocks > cap) blocks = cap;
  focal_elementwise_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(y_true, y_pred, n, normalizer, alpha, gamma, label_smoothing, out);
  B200_LAUNCH_CHECK();
  return B200_OK;
}

extern "C" size_t b200_focal_box_workspace_bytes(int num_levels, const unsigned long long* anchors_per_level, int C) {
  unsigned long long elems[EL_MAX_LEVELS];
  int cta_base[EL_MAX_LEVELS + 1];
  if (num_levels < 1 || num_levels > EL_MAX_LEVELS) return 0;
  for (int l = 0; l < num_levels; ++l) elems[l] = anchors_per_level[l] * (unsigned long long)C;
  const int n = el_cta_plan(num_levels, elems, cta_base);
  return b200_align_up(sizeof(double) * 3 * (size_t)n, 256);
}

// anchors_per_level[l] = B*H_l*W_l*A of THIS call (local shard); sums_out: device double[2L+1]
static int el_partial_sums_impl(int num_levels, const unsigned long long* anchors_per_level, int C,
                                const float* const true_boxes[], const float* const true_classes_dense[],
                                const int32_t* const true_class_index[], const unsigned char* const true_masks[],
                                const float* const pred_boxes[], const float* const pred_classes[], float alpha, float gamma,
                                float delta, float label_smoothing, double* sums_out, void* workspace, size_t workspace_bytes,
                                void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  B200_REQUIRE(num_levels >= 1 && num_levels <= EL_MAX_LEVELS && C >= 1, B200_ERR_BAD_ARG, "b200_focal_box_partial_sums: bad level count / classes");
  B200_REQUIRE(anchors_per_level && true_boxes && (true_classes_dense || true_class_index) && true_masks && pred_boxes && pred_classes && sums_out,
               B200_ERR_BAD_ARG, "b200_focal_box_partial_sums: null argument");
  // the class targets of a level: the one-hot tensor, or (sparse-target mode) one class id per anchor
  const void* true_classes[EL_MAX_LEVELS];
  for (int l = 0; l < EL_MAX_LEVELS; ++l)
    true_classes[l] = l < num_levels ? (true_classes_dense ? (const void*)true_classes_dense[l] : (const void*)true_class_index[l]) : nullptr;
  ElParams p;
  p.C = C;
  unsigned long long elems[EL_MAX_LEVELS];
  p.num_levels = num_levels;
  for (int l = 0; l < EL_MAX_LEVELS; ++l) {
    if (l < num_levels) {
      // either half of a level may be absent (stand-alone FocalLoss / BoxLoss calls)
      const bool has_cls = true_classes[l] && pred_classes[l];
      const bool has_box = true_boxes[l] && pred_boxes[l] && true_masks[l];
      B200_REQUIRE(has_cls || has_box, B200_ERR_BAD_ARG, "b200_focal_box_partial_sums: null level %d", l);
      const uintptr_t al = reinterpret_cast<uintptr_t>(true_boxes[l]) | reinterpret_cast<uintptr_t>(true_classes[l]) |
                           reinterpret_cast<uintptr_t>(pred_boxes[l]) | reinterpret_cast<uintptr_t>(pred_classes[l]);
      B200_REQUIRE((al & 15) == 0, B200_ERR_BAD_ARG, "b200_focal_box_partial_sums: level %d tensors must be 16-byte aligned", l);
      elems[l] = has_cls ? anchors_per_level[l] * (unsigned long long)C : 0ull;
      p.cls_pred[l] = reinterpret_cast<const float4*>(pred_classes[l]);
      p.cls_true[l] = true_classes_dense ? reinterpret_cast<const float4*>(true_classes[l]) : nullptr;
      p.cls_index[l] = true_classes_dense ? nullptr : reinterpret_cast<const int32_t*>(true_classes[l]);
      p.cls_vec[l] = elems[l] / 4;
      p.cls_tail[l] = (int)(elems[l] - p.cls_vec[l] * 4);
      p.cls_pred_tail[l] = pred_classes[l] + p.cls_vec[l] * 4;
      p.cls_true_tail[l] = true_classes_dense ? true_classes_dense[l] + p.cls_vec[l] * 4 : nullptr;
      p.box_pred[l] = reinterpret_cast<const float4*>(pred_boxes[l]);
      p.box_true[l] = reinterpret_cast<const float4*>(true_boxes[l]);
      p.mask[l] = true_masks[l];
      p.anchors[l] = has_box ? anchors_per_level[l] : 0ull;
    } else {
      elems[l] = 0; p.cls_pred[l] = p.cls_true[l] = nullptr; p.cls_index[l] = nullptr; p.cls_vec[l] = 0; p.cls_tail[l] = 0;
      p.cls_pred_tail[l] = p.cls_true_tail[l] = nullptr; p.box_pred[l] = p.box_true[l] = nullptr; p.mask[l] = nullptr; p.anchors[l] = 0;
    }
  }
  unsigned long long plan[EL_MAX_LEVELS];
  for (int l = 0; l < EL_MAX_LEVELS; ++l) plan[l] = elems[l] > p.anchors[l] * 4ull ? elems[l] : p.anchors[l] * 4ull;
  const int n_cta = el_cta_plan(num_levels, plan, p.cta_base);
  const size_t need = b200_align_up(sizeof(double) * 3 * (size_t)n_cta, 256);
  B200_REQUIRE(workspace && workspace_bytes >= need, B200_ERR_WORKSPACE, "b200_focal_box_partial_sums: workspace %zu < required %zu", workspace_bytes, need);
  p.alpha = alpha; p.gamma = gamma; p.delta = delta; p.label_smoothing = label_smoothing;
  p.partials = static_cast<double*>(workspace);
  B200_CUDA(cudaMemsetAsync(sums_out, 0, sizeof(double) * (2 * num_levels + 1), stream));
  if (gamma == 1.5f) focal_box_partials_kernel<true><<<n_cta, EL_THREADS, 0, stream>>>(p);
  else focal_box_partials_kernel<false><<<n_cta, EL_THREADS, 0, stream>>>(p);
  B200_LAUNCH_CHECK();
  ElReduce r;
  r.partials = p.partials; r.num_levels = num_levels; r.sums = sums_out;
  for (int l = 0; l <= EL_MAX_LEVELS; ++l) r.cta_base[l] = p.cta_base[l];
  focal_box_reduce_kernel<<<num_levels, 256, 0, stream>>>(r);
  B200_LAUNCH_CHECK();
  return B200_OK;
}

extern "C" int b200_focal_box_partial_sums(int num_levels, const unsigned long long* anchors_per_level, int C,
                                           const float* const true_boxes[], const float* const true_classes[],
                                           const unsigned char* const true_masks[], const float* const pred_boxes[],
                                           const float* const pred_classes[], float alpha, float gamma, float delta,
                                           float label_smoothing, double* sums_out, void* workspace,
                                           size_t workspace_bytes, void* stream_) {
  B200_REQUIRE(true_classes, B200_ERR_BAD_ARG, "b200_focal_box_partial_sums: null argument");
  return el_partial_sums_impl(num_levels, anchors_per_level, C, true_boxes, true_classes, nullptr, true_masks, pred_boxes,
                              pred_classes, alpha, gamma, delta, label_smoothing, sums_out, workspace, workspace_bytes, stream_);
}

// Sparse-target mode (SURVEY §8f N3): true_class_index[l] (B,H,W,A) int32 = the class id whose one-hot row
// generate_targets would have written (0 for unmatched anchors; out-of-range ids = all-zero row).
extern "C" int b200_focal_box_partial_sums_indexed(int num_levels, const unsigned long long* anchors_per_level, int C,
                                                   const float* const true_boxes[], const int32_t* const true_class_index[],
                                                   const unsigned char* const true_masks[], const float* const pred_boxes[],
                                                   const float* const pred_classes[], float alpha, float gamma, float delta,
                                                   float label_smoothing, double* sums_out, void* workspace,
                                                   size_t workspace_bytes, void* stream_) {
  B200_REQUIRE(true_class_index, B200_ERR_BAD_ARG, "b200_focal_box_partial_sums_indexed: null argument");
  return el_partial_sums_impl(num_levels, anchors_per_level, C, true_boxes, nullptr, true_class_index, true_masks, pred_boxes,
                              pred_classes, alpha, gamma, delta, label_smoothing, sums_out, workspace, workspace_bytes, stream_);
}

// numel_per_level[l] = GLOBAL element count B_global*H*W*A*C of level l (the Keras mean divisor)
int b200_fill_exchange(B200Exchange& x, int rank, int world, void* const mailboxes[], const char* who);

static int el_finalize_impl(int num_levels, double* sums, const double* numel_per_level_host, float* out_parts, float* out_loss,
                            float* out_num_positives, const B200Exchange& x, void* stream) {
  B200_REQUIRE(num_levels >= 1 && num_levels <= EL_MAX_LEVELS && sums && numel_per_level_host && out_loss, B200_ERR_BAD_ARG,
               "b200_focal_box_finalize: bad argument");
  ElFinalize f;
  f.sums = sums; f.num_levels = num_levels; f.parts = out_parts; f.loss = out_loss; f.num_pos = out_num_positives;
  f.xchg = x;
  for (int l = 0; l < EL_MAX_LEVELS; ++l) f.numel[l] = l < num_levels ? numel_per_level_host[l] : 1.0;
  focal_box_finalize_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(f);
  B200_LAUNCH_CHECK();
  return B200_OK;
}

extern "C" int b200_focal_box_finalize(int num_levels, const double* sums, const double* numel_per_level_host,
                                       float* out_parts, float* out_loss, float* out_num_positives, void* stream) {
  B200Exchange x;
  b200_fill_exchange(x, 0, 1, nullptr, "b200_focal_box_finalize");
  return el_finalize_impl(num_levels, const_cast<double*>(sums), numel_per_level_host, out_parts, out_loss, out_num_positives, x, stream);
}

// Data-parallel finalize: `sums` holds THIS rank's partial sums on entry and the global sums on return (all-reduced
// inside the kernel through the peer mailboxes); numel_per_level_host = GLOBAL element counts.
extern "C" int b200_focal_box_finalize_dp(int num_levels, double* sums, const double* numel_per_level_host, float* out_parts,
                                          float* out_loss, float* out_num_positives, int rank, int world,
                                          void* const mailboxes[], void* stream) {
  B200Exchange x;
  const int rc = b200_fill_exchange(x, rank, world, mailboxes, "b200_focal_box_finalize_dp");
  if (rc != B200_OK) return rc;
  return el_finalize_impl(num_levels, sums, numel_per_level_host, out_parts, out_loss, out_num_positives, x, stream);
}

// d loss / d pred_classes[l] and d loss / d pred_boxes[l] (either array entry may be NULL).  `sums` is the device
// array b200_focal_box_partial_sums produced (after the all-reduce, if any); numel_per_level_host as in finalize.
static int el_grad_impl(int num_levels, const unsigned long long* anchors_per_level, int C,
                        const float* const true_boxes[], const float* const true_classes[],
                        const int32_t* const true_class_index[],
                        const float* const pred_boxes[], const float* const pred_classes[], float alpha,
                        float gamma, float delta, float label_smoothing, const double* sums,
                        const double* numel_per_level_host, float* const grad_boxes[],
                        float* const grad_classes[], void* stream) {
  B200_REQUIRE(num_levels >= 1 && num_levels <= EL_MAX_LEVELS && C >= 1 && anchors_per_level && sums && numel_per_level_host,
               B200_ERR_BAD_ARG, "b200_focal_box_grad: bad argument");
  B200_REQUIRE(!true_class_index || C >= 4, B200_ERR_UNSUPPORTED, "b200_focal_box_grad_indexed: needs classes_num >= 4");
  ElGradParams p;
  p.C = C;
  unsigned long long plan[EL_MAX_LEVELS];
  p.num_levels = num_levels;
  for (int l = 0; l < EL_MAX_LEVELS; ++l) {
    p.cls_pred[l] = p.cls_true[l] = nullptr; p.cls_grad[l] = nullptr; p.box_pred[l] = p.box_true[l] = nullptr; p.box_grad[l] = nullptr;
    p.cls_index[l] = nullptr;
    p.cls_vec[l] = 0; p.cls_tail[l] = 0; p.anchors[l] = 0; p.numel[l] = 1.0; plan[l] = 0;
    if (l >= num_levels) continue;
    p.numel[l] = numel_per_level_host[l];
    if (grad_classes && grad_classes[l]) {
      const void* tcl = true_class_index ? (const void*)true_class_index[l] : (true_classes ? (const void*)true_classes[l] : nullptr);
      B200_REQUIRE(tcl && pred_classes && pred_classes[l], B200_ERR_BAD_ARG, "b200_focal_box_grad: null class tensors at level %d", l);
      const unsigned long long n = anchors_per_level[l] * (unsigned long long)C;
      const uintptr_t al = (true_class_index ? 0 : reinterpret_cast<uintptr_t>(tcl)) | reinterpret_cast<uintptr_t>(pred_classes[l]) | reinterpret_cast<uintptr_t>(grad_classes[l]);
      B200_REQUIRE((al & 15) == 0, B200_ERR_BAD_ARG, "b200_focal_box_grad: level %d class tensors must be 16-byte aligned", l);
      p.cls_pred[l] = reinterpret_cast<const float4*>(pred_classes[l]);
      p.cls_true[l] = true_class_index ? nullptr : reinterpret_cast<const float4*>(tcl);
      p.cls_index[l] = true_class_index ? true_class_index[l] : nullptr;
      p.cls_grad[l] = reinterpret_cast<float4*>(grad_classes[l]);
      p.cls_vec[l] = n / 4ull;
      p.cls_tail[l] = (int)(n - p.cls_vec[l] * 4ull);
      plan[l] = n;
    }
    if (grad_boxes && grad_boxes[l]) {
      B200_REQUIRE(true_boxes && pred_boxes && true_boxes[l] && pred_boxes[l], B200_ERR_BAD_ARG, "b200_focal_box_grad: null box tensors at level %d", l);
      const uintptr_t al = reinterpret_cast<uintptr_t>(true_boxes[l]) | reinterpret_cast<uintptr_t>(pred_boxes[l]) | reinterpret_cast<uintptr_t>(grad_boxes[l]);
      B200_REQUIRE((al & 15) == 0, B200_ERR_BAD_ARG, "b200_focal_box_grad: level %d box tensors must be 16-byte aligned", l);
      p.box_pred[l] = reinterpret_cast<const float4*>(pred_boxes[l]);
      p.box_true[l] = reinterpret_cast<const float4*>(true_boxes[l]);
      p.box_grad[l] = reinterpret_cast<float4*>(grad_boxes[l]);
      p.anchors[l] = anchors_per_level[l];
      if (plan[l] < anchors_per_level[l] * 4ull) plan[l] = anchors_per_level[l] * 4ull;
    }
    if (plan[l] == 0) plan[l] = 4;
  }
  const int n_cta = el_cta_plan(num_levels, plan, p.cta_base);
  p.alpha = alpha; p.gamma = gamma; p.delta = delta; p.label_smoothing = label_smoothing; p.sums = sums;
  focal_box_grad_kernel<<<n_cta, EL_THREADS, 0, (cudaStream_t)stream>>>(p);
  B200_LAUNCH_CHECK();
  return B200_OK;
}

extern "C" int b200_focal_box_grad(int num_levels, const unsigned long long* anchors_per_level, int C,
                                   const float* const true_boxes[], const float* const true_classes[],
                                   const float* const pred_boxes[], const float* const pred_classes[], float alpha,
                                   float gamma, float delta, float label_smoothing, const double* sums,
                                   const double* numel_per_level_host, float* const grad_boxes[],
                                   float* const grad_classes[], void* stream) {
  return el_grad_impl(num_levels, anchors_per_level, C, true_boxes, true_classes, nullptr, pred_boxes, pred_classes, alpha, gamma,
                      delta, label_smoothing, sums, numel_per_level_host, grad_boxes, grad_classes, stream);
}

// Sparse-target mode of the backward pass: true_class_index[l] (B,H,W,A) int32 class ids, as
// b200_focal_box_partial_sums_indexed takes them (the one-hot row is rebuilt in registers).
extern "C" int b200_focal_box_grad_indexed(int num_levels, const unsigned long long* anchors_per_level, int C,
                                           const float* const true_boxes[], const int32_t* const true_class_index[],
                                           const float* const pred_boxes[], const float* const pred_classes[], float alpha,
                                           float gamma, float delta, float label_smoothing, const double* sums,
                                           const double* numel_per_level_host, float* const grad_boxes[],
                                           float* const grad_classes[], void* stream) {
  B200_REQUIRE(true_class_index, B200_ERR_BAD_ARG, "b200_focal_box_grad_indexed: null argument");
  return el_grad_impl(num_levels, anchors_per_level, C, true_boxes, nullptr, true_class_index, pred_boxes, pred_classes, alpha,
                      gamma, delta, label_smoothing, sums, numel_per_level_host, grad_boxes, grad_classes, stream);
}

// ---- loss and gradient from box lists, stage 2 (SURVEY §8f N3 + N1) --------------------------------------------------
// One pass over the heads after b200_effdet_loss_from_boxes_match (effdet.cu) has left the matched GT row of every anchor
// in the workspace: the class of an anchor is gt_classes[match] (0 = background when unmatched), its box target is
// encoded in registers from the rebuilt anchor and the GT box.  The focal and Huber terms go to per-CTA partials
// {focal_l, huber_l, 0} (the positives are the match stage's), the gradients — the arithmetic of focal_box_grad_kernel on
// the same targets, so the same bits — are written when their pointers are given.
#define EFB_MAX_CTAS 16384   // cap of the CTA plan: keeps the workspace size independent of the device

struct EfbParams {
  EfLevels lv;
  int B, C;
  const float* gt_boxes;       // [total,4] y1,x1,y2,x2
  const int32_t* gt_classes;   // [total]
  const int32_t* match;        // per anchor: row of gt_boxes or -1; level l at B*anchor_base[l]
  const float4* cls_pred[EL_MAX_LEVELS]; float4* cls_grad[EL_MAX_LEVELS];
  const float4* box_pred[EL_MAX_LEVELS]; float4* box_grad[EL_MAX_LEVELS];
  unsigned long long cls_vec[EL_MAX_LEVELS];
  int cls_tail[EL_MAX_LEVELS];
  unsigned long long anchors[EL_MAX_LEVELS];   // B*H*W*A
  double numel[EL_MAX_LEVELS];
  int cta_base[EL_MAX_LEVELS + 1];
  float alpha, gamma, delta, label_smoothing;
  const double* sums;   // sums[2L] = positives (after the caller's all-reduce)
  double* partials;     // [n_cta, 3]
};

// the class id whose one-hot row generate_targets writes for anchor a (anc:131-133: class 0 when unmatched)
__device__ __forceinline__ int efb_class(const EfbParams& p, const int32_t* match, unsigned long long a) {
  const int m = __ldg(match + a);
  return m >= 0 ? __ldg(p.gt_classes + m) : 0;
}

__global__ void __launch_bounds__(EL_THREADS) effdet_loss_from_boxes_kernel(EfbParams p) {
  __shared__ double s_red[EL_THREADS / 32][2];
  int l = 0;
#pragma unroll
  for (int k = 1; k < EL_MAX_LEVELS; ++k) if (k < p.lv.num_levels && (int)blockIdx.x >= p.cta_base[k]) l = k;
  const int ncta = p.cta_base[l + 1] - p.cta_base[l];
  const int cta = blockIdx.x - p.cta_base[l];
  const unsigned long long stride = (unsigned long long)ncta * EL_THREADS;
  const float npos = (float)p.sums[2 * p.lv.num_levels] + 1.0f;
  const float cs = (float)(1.0 / ((double)npos * p.numel[l]));
  const float bs = 50.0f / (4.0f * npos);
  const int32_t* __restrict__ match = p.match + (size_t)p.B * p.lv.anchor_base[l];
  const int C = p.C;
  // class half: flat float4 walk over the logits; a float4 straddles at most two anchors (C >= 4)
  float f0 = 0.f, f1 = 0.f;
  double focal = 0.0;
  int it = 0;
  const float4* __restrict__ cp = p.cls_pred[l];
  float4* __restrict__ cg = p.cls_grad[l];
  const unsigned long long nv = p.cls_vec[l];
#pragma unroll 2
  for (unsigned long long i = (unsigned long long)cta * EL_THREADS + threadIdx.x; i < nv; i += stride) {
    const float4 x = __ldcs(cp + i);
    const unsigned long long e = i * 4ull, a0 = e / (unsigned long long)C;
    const int c0 = (int)(e - a0 * (unsigned long long)C);
    const int id0 = efb_class(p, match, a0);
    const int id1 = (c0 + 3 >= C) ? efb_class(p, match, a0 + 1) : 0;
    float yy[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int c = c0 + k;
      yy[k] = (c < C) ? ((c == id0) ? 1.0f : 0.0f) : ((c - C == id1) ? 1.0f : 0.0f);   // ids outside [0, C): zero row
    }
    float v0, v1, v2, v3;
    float4 g;
    g.x = cs * el_focal_value_grad(yy[0], x.x, p.alpha, p.gamma, p.label_smoothing, v0);
    g.y = cs * el_focal_value_grad(yy[1], x.y, p.alpha, p.gamma, p.label_smoothing, v1);
    g.z = cs * el_focal_value_grad(yy[2], x.z, p.alpha, p.gamma, p.label_smoothing, v2);
    g.w = cs * el_focal_value_grad(yy[3], x.w, p.alpha, p.gamma, p.label_smoothing, v3);
    if (cg) __stcs(cg + i, g);
    f0 += v0 + v1;
    f1 += v2 + v3;
    if ((++it & 63) == 0) { focal += (double)f0 + (double)f1; f0 = f1 = 0.f; }
  }
  if (cta == 0 && (int)threadIdx.x < p.cls_tail[l]) {
    const unsigned long long e = nv * 4ull + threadIdx.x, a = e / (unsigned long long)C;
    const float yt = ((int)(e - a * (unsigned long long)C) == efb_class(p, match, a)) ? 1.0f : 0.0f;
    float v;
    const float g = cs * el_focal_value_grad(yt, reinterpret_cast<const float*>(cp)[e], p.alpha, p.gamma, p.label_smoothing, v);
    if (cg) reinterpret_cast<float*>(cg)[e] = g;
    f0 += v;
  }
  focal += (double)f0 + (double)f1;
  // box half: one anchor per thread, the target encoded from the rebuilt anchor and the matched GT box
  float hub = 0.f;
  const unsigned long long na = p.anchors[l];
  const unsigned int api = (unsigned int)p.lv.anc_per_img[l];
  float4* __restrict__ bg = p.box_grad[l];
  for (unsigned long long a = (unsigned long long)cta * EL_THREADS + threadIdx.x; a < na; a += stride) {
    const float4 o = __ldcs(p.box_pred[l] + a);
    const int m = __ldg(match + a);
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
    if (m >= 0) {
      const int rin = (int)(a % api);
      int y, x, an_i;
      ef_split(p.lv, l, rin, y, x, an_i);
      const AnchorBox an = ef_anchor(p.lv, l, y, x, an_i);
      const float4 q = __ldg(reinterpret_cast<const float4*>(p.gt_boxes) + m);
      t = ef_encode_box(an.y1, an.x1, an.y2, an.x2, q.x, q.y, q.z, q.w);
    }
    hub += el_huber(t.x, o.x, p.delta) + el_huber(t.y, o.y, p.delta) + el_huber(t.z, o.z, p.delta) + el_huber(t.w, o.w, p.delta);
    if (bg) __stcs(bg + a, make_float4(bs * el_huber_grad(t.x, o.x, p.delta), bs * el_huber_grad(t.y, o.y, p.delta),
                                       bs * el_huber_grad(t.z, o.z, p.delta), bs * el_huber_grad(t.w, o.w, p.delta)));
  }
  const double v0 = warp_sum_d(focal), v1 = warp_sum_d((double)hub);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { s_red[warp][0] = v0; s_red[warp][1] = v1; }
  __syncthreads();
  if (threadIdx.x < 3) {
    double s = 0.0;
    if (threadIdx.x < 2)
      for (int w = 0; w < EL_THREADS / 32; ++w) s += s_red[w][threadIdx.x];
    p.partials[(size_t)blockIdx.x * 3 + threadIdx.x] = s;   // {focal_l, huber_l, 0}
  }
}

// workspace: [match: int32 per anchor of the batch][partials: 3 doubles per CTA]
static size_t efb_match_bytes(int anchors_per_image, int B) {
  return b200_align_up(sizeof(int32_t) * (size_t)anchors_per_image * (size_t)B, 256);
}

size_t efb_workspace_bytes(int num_levels, int anchors_per_image, int B) {
  return efb_match_bytes(anchors_per_image, B) + b200_align_up(sizeof(double) * 3 * (size_t)(EFB_MAX_CTAS + num_levels), 256);
}

extern "C" size_t b200_effdet_loss_from_boxes_workspace_bytes(int num_levels, const int32_t* hw, int A, int B) {
  EfLevels lv;
  if (!hw || B < 0) return 0;
  const int n_img = ef_fill_levels(lv, num_levels, hw, A, nullptr);
  return n_img < 0 ? 0 : efb_workspace_bytes(num_levels, n_img, B);
}

extern "C" int b200_effdet_loss_from_boxes_grad(int num_levels, const int32_t* hw, int A, const float* table_dev, int C, int B,
                                                const float* gt_boxes, const int32_t* gt_classes, int total_boxes,
                                                const float* const pred_boxes[], const float* const pred_classes[], float alpha,
                                                float gamma, float delta, float label_smoothing,
                                                const double* numel_per_level_host, double* sums, float* const grad_boxes[],
                                                float* const grad_classes[], void* workspace, size_t workspace_bytes,
                                                void* stream_) {
  const char* who = "b200_effdet_loss_from_boxes_grad";
  cudaStream_t stream = (cudaStream_t)stream_;
  EfbParams p;
  B200_REQUIRE(hw && table_dev && pred_boxes && pred_classes && numel_per_level_host && sums, B200_ERR_BAD_ARG, "%s: null argument", who);
  const int n_img = ef_fill_levels(p.lv, num_levels, hw, A, table_dev);
  B200_REQUIRE(n_img >= 0, B200_ERR_BAD_ARG, "%s: bad level spec", who);
  B200_REQUIRE(C >= 4, B200_ERR_UNSUPPORTED, "%s: needs classes_num >= 4 (got %d)", who, C);
  B200_REQUIRE(B >= 0 && total_boxes >= 0, B200_ERR_BAD_ARG, "%s: negative batch or box count", who);
  B200_REQUIRE(total_boxes == 0 || (gt_boxes && gt_classes), B200_ERR_BAD_ARG, "%s: null gt_boxes / gt_classes", who);
  B200_REQUIRE((reinterpret_cast<uintptr_t>(gt_boxes) & 15) == 0, B200_ERR_BAD_ARG, "%s: gt_boxes not 16-byte aligned", who);
  unsigned long long plan[EL_MAX_LEVELS];
  for (int l = 0; l < EL_MAX_LEVELS; ++l) {
    p.cls_pred[l] = nullptr; p.cls_grad[l] = nullptr; p.box_pred[l] = nullptr; p.box_grad[l] = nullptr;
    p.cls_vec[l] = 0; p.cls_tail[l] = 0; p.anchors[l] = 0; p.numel[l] = 1.0; plan[l] = 0;
    if (l >= num_levels) continue;
    B200_REQUIRE(pred_boxes[l] && pred_classes[l], B200_ERR_BAD_ARG, "%s: null prediction at level %d", who, l);
    B200_REQUIRE(!grad_boxes || grad_boxes[l], B200_ERR_BAD_ARG, "%s: null grad_boxes at level %d", who, l);
    B200_REQUIRE(!grad_classes || grad_classes[l], B200_ERR_BAD_ARG, "%s: null grad_classes at level %d", who, l);
    const uintptr_t al = reinterpret_cast<uintptr_t>(pred_boxes[l]) | reinterpret_cast<uintptr_t>(pred_classes[l]) |
                         (grad_boxes ? reinterpret_cast<uintptr_t>(grad_boxes[l]) : 0) |
                         (grad_classes ? reinterpret_cast<uintptr_t>(grad_classes[l]) : 0);
    B200_REQUIRE((al & 15) == 0, B200_ERR_BAD_ARG, "%s: level %d tensors must be 16-byte aligned", who, l);
    B200_REQUIRE(numel_per_level_host[l] > 0.0, B200_ERR_BAD_ARG, "%s: numel of level %d must be positive", who, l);
    const unsigned long long na = (unsigned long long)B * (unsigned long long)p.lv.anc_per_img[l], n = na * (unsigned long long)C;
    p.cls_pred[l] = reinterpret_cast<const float4*>(pred_classes[l]);
    p.cls_grad[l] = grad_classes ? reinterpret_cast<float4*>(grad_classes[l]) : nullptr;
    p.box_pred[l] = reinterpret_cast<const float4*>(pred_boxes[l]);
    p.box_grad[l] = grad_boxes ? reinterpret_cast<float4*>(grad_boxes[l]) : nullptr;
    p.cls_vec[l] = n / 4ull;
    p.cls_tail[l] = (int)(n - p.cls_vec[l] * 4ull);
    p.anchors[l] = na;
    p.numel[l] = numel_per_level_host[l];
    plan[l] = n > na * 4ull ? n : na * 4ull;
    if (plan[l] == 0) plan[l] = 4;
  }
  const size_t need = efb_workspace_bytes(num_levels, n_img, B);
  B200_REQUIRE(workspace && workspace_bytes >= need, B200_ERR_WORKSPACE, "%s: workspace %zu < required %zu", who, workspace_bytes, need);
  B200_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, B200_ERR_BAD_ARG, "%s: workspace not 256-byte aligned", who);
  if (B == 0) return B200_OK;   // the match stage left sums[0..2L) at zero
  p.B = B; p.C = C;
  p.gt_boxes = gt_boxes; p.gt_classes = gt_classes;
  unsigned char* wsb = static_cast<unsigned char*>(workspace);
  p.match = reinterpret_cast<const int32_t*>(wsb);
  p.partials = reinterpret_cast<double*>(wsb + efb_match_bytes(n_img, B));
  p.alpha = alpha; p.gamma = gamma; p.delta = delta; p.label_smoothing = label_smoothing; p.sums = sums;
  const int budget = b200_sm_count() * 64;
  const int n_cta = el_cta_plan_budget(num_levels, plan, p.cta_base, budget < EFB_MAX_CTAS ? budget : EFB_MAX_CTAS);
  effdet_loss_from_boxes_kernel<<<n_cta, EL_THREADS, 0, stream>>>(p);
  B200_LAUNCH_CHECK();
  ElReduce r;
  r.partials = p.partials; r.num_levels = num_levels; r.sums = sums;
  for (int l = 0; l <= EL_MAX_LEVELS; ++l) r.cta_base[l] = p.cta_base[l];
  focal_box_reduce_kernel<<<num_levels, 256, 0, stream>>>(r);   // sums[0..2L); adds the partials' 0 to sums[2L]
  B200_LAUNCH_CHECK();
  return B200_OK;
}
