// map.cu — per-image mAP, the step right after NMS in test_step (SURVEY §8f N2).
//
// Replaces utils/mAP.py:3-125 (Get_TPFP / Get_AP / Get_mAP_one), which the reference reaches through
// tf.numpy_function (a GIL round trip with a Python loop over the classes; yolo_v4/model.py:377, edt:166).
// One CTA per image, fp64 like the NumPy original.  Per class: compact the class's predictions and ground truth
// (order preserved), one thread per ground-truth box finds its arg-max-IoU prediction (first maximum) and marks it
// a true positive when IoU >= thresh, a rank sort orders the predictions by score (descending; equal scores in
// reversed index order, as a stable argsort followed by [::-1] gives), and one thread walks the list to build the
// reference's precision/recall arrays, their envelope and the AP sum exactly as written (including its swapped
// mrec/mpre naming, mAP.py:88-99).
//
// Two input forms share that per-class body (map_image): packed rows with host-known per-image maxima (map_kernel,
// b200_map_per_image), and the padded NMS output [B,K] with device counts plus ground-truth box lists
// (map_padded_kernel, b200_map_padded).  The ground truth of an image is walked in chunks, so the padded form needs no
// per-image maximum: shared memory depends on K alone, and the call never waits for the host.
#include "common.cuh"
#include "nms.cuh"

#define MAP_THREADS 256
#define MAP_GT_CHUNK 1024   // ground-truth rows compacted per pass in the padded form

// ---- per-class body shared by both kernels ------------------------------------------------------------------------
// A source exposes, for the image of the CTA: pr_is(i, c) / gt_is(i, c) (row i has class c), pr_box / gt_box (x1, y1,
// x2, y2 as doubles of the stored floats) and pr_score(i).

// ordered compaction of rows [base, base + n) for which is_c(row) holds into dst (row numbers); returns the count
// (block-uniform)
template <typename F>
__device__ __forceinline__ int map_compact(int base, int n, F is_c, int* dst, int* s_warp) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int run = 0;
  for (int i0 = 0; i0 < n; i0 += MAP_THREADS) {
    const int i = i0 + tid;
    const bool f = (i < n) && is_c(base + i);
    const uint32_t bal = __ballot_sync(0xffffffffu, f);
    if (lane == 0) s_warp[warp] = __popc(bal);
    __syncthreads();
    int off = run;
    for (int w = 0; w < warp; ++w) off += s_warp[w];
    if (f) dst[off + __popc(bal & ((1u << lane) - 1u))] = base + i;
    int tot = 0;
    for (int w = 0; w < MAP_THREADS / 32; ++w) tot += s_warp[w];
    run += tot;
    __syncthreads();
  }
  return run;
}

// each listed ground-truth box claims its arg-max-IoU prediction of the class
template <typename S>
__device__ __forceinline__ void map_claim(const S& s, const int* s_gi, int ng, const int* s_pi, int np, int* s_tp, double thresh) {
  for (int g = threadIdx.x; g < ng; g += MAP_THREADS) {
    double gx1, gy1, gx2, gy2;
    s.gt_box(s_gi[g], gx1, gy1, gx2, gy2);
    const double ga = (gx2 - gx1) * (gy2 - gy1);
    int best = 0;
    double bv = 0.0;
    for (int q = 0; q < np; ++q) {
      double px1, py1, px2, py2;
      s.pr_box(s_pi[q], px1, py1, px2, py2);
      const double iw = fmax(fmin(gx2, px2) - fmax(gx1, px1), 0.0), ih = fmax(fmin(gy2, py2) - fmax(gy1, py1), 0.0);
      const double inter = iw * ih;
      const double iou = inter / (ga + (px2 - px1) * (py2 - py1) - inter);
      // np.argmax (mAP.py:53): the first maximal index, and a NaN (0/0: zero-area boxes) counts as maximal — the
      // first NaN freezes the choice, and `NaN >= thresh` is False, so that ground-truth box claims nothing
      if (q == 0 || (bv == bv && (iou > bv || iou != iou))) { bv = iou; best = q; }
    }
    if (bv >= thresh) s_tp[best] = 1;
  }
}

struct MapSmem {
  double* a; double* b;   // [cap_p + 2] "mrec" (precision list), "mpre" (recall list)
  int* pi; int* tp; int* sorted;   // [cap_p] prediction rows of the class, tp flag per row, tp flags in sorted order
  int* gi;                // [cap_g] ground-truth rows of the class
};

__device__ __forceinline__ MapSmem map_smem_carve(unsigned char* base, int cap_p, int cap_g) {
  MapSmem m;
  m.a = reinterpret_cast<double*>(base);
  m.b = m.a + cap_p + 2;
  m.pi = reinterpret_cast<int*>(m.b + cap_p + 2);
  m.gi = m.pi + cap_p;
  m.tp = m.gi + cap_g;
  m.sorted = m.tp + cap_p;
  return m;
}

static size_t map_smem_bytes(int cap_p, int cap_g) {
  return sizeof(double) * 2 * (size_t)(cap_p + 2) + sizeof(int) * (3 * (size_t)cap_p + cap_g);
}

// mAP of one image: np_all predictions, ng_all ground-truth rows walked gt_chunk at a time.  The value is valid on
// thread 0.
template <typename S>
__device__ __forceinline__ double map_image(const S& s, int np_all, int ng_all, int gt_chunk, int class_num, double thresh, const MapSmem& m) {
  __shared__ int s_warp[MAP_THREADS / 32];
  // in shared memory: registers would be saved around every call of the fp64 division
  __shared__ double s_total;
  __shared__ int s_ng;
  if (ng_all == 0) return 0.0;   // every class has AP 0
  const int tid = threadIdx.x;
  if (tid == 0) s_total = 0.0;
  for (int c = 0; c < class_num; ++c) {
    const int np_c = map_compact(0, np_all, [s, c](int i) { return s.pr_is(i, c); }, m.pi, s_warp);
    if (np_c == 0) continue;   // AP = 0 (mAP.py:29-30 -> empty tp list)
    for (int i = tid; i < np_c; i += MAP_THREADS) m.tp[i] = 0;
    if (tid == 0) s_ng = 0;   // the previous class's readers are past the barriers of the compaction above
    for (int g0 = 0; g0 < ng_all; g0 += gt_chunk) {
      const int n = map_compact(g0, min(gt_chunk, ng_all - g0), [s, c](int i) { return s.gt_is(i, c); }, m.gi, s_warp);
      map_claim(s, m.gi, n, m.pi, np_c, m.tp, thresh);
      if (tid == 0) s_ng += n;
      __syncthreads();   // the claims of this chunk are in, its rows may be overwritten
    }
    const int ng_c = s_ng;   // ng_all > 0: the loop above ran and ended on a barrier
    if (ng_c == 0) continue;   // AP = 0
    // ---- rank sort by score, descending; ties: higher original position first ----
    for (int i = tid; i < np_c; i += MAP_THREADS) {
      const float si = s.pr_score(m.pi[i]);
      int rank = 0;
      for (int j = 0; j < np_c; ++j) {
        const float sj = s.pr_score(m.pi[j]);
        rank += (sj > si || (sj == si && j > i)) ? 1 : 0;
      }
      m.sorted[rank] = m.tp[i];
    }
    __syncthreads();
    // ---- AP exactly as mAP.py:74-99 ----
    if (tid == 0) {
      double sum = 0.0;
      m.a[0] = 0.0; m.b[0] = 0.0;
      for (int i = 0; i < np_c; ++i) {
        if (m.sorted[i] == 1) sum += 1.0;
        m.a[i + 1] = sum / (double)(i + 1);   // "precision_list" -> mrec
        m.b[i + 1] = sum / (double)ng_c;      // "recall_list"    -> mpre
      }
      m.a[np_c + 1] = 1.0; m.b[np_c + 1] = 0.0;
      for (int i = np_c + 1; i > 0; --i) m.b[i - 1] = fmax(m.b[i - 1], m.b[i]);
      double ap = 0.0;
      for (int i = 0; i <= np_c; ++i)
        if (m.a[i + 1] != m.a[i]) ap += (m.a[i + 1] - m.a[i]) * m.b[i + 1];
      s_total += ap;
    }
    __syncthreads();
  }
  return s_total / (double)class_num;
}

// ---- packed rows: gt [total,5] x1,y1,x2,y2,class ; pred [total,6] x1,y1,x2,y2,class,score -------------------------
struct MapParams {
  const float* gt; const int32_t* gt_off;   // [total_gt,5] ; [B+1]
  const float* pr; const int32_t* pr_off;   // [total_pr,6] ; [B+1]
  int class_num; double thresh;
  int cap_p, cap_g;                         // per-image capacities of the shared lists
  double* out;                              // [B]
};

struct MapRowsSrc {
  const float* gt; const float* pr;
  __device__ bool pr_is(int i, int c) const { return (double)pr[6 * (size_t)i + 4] == (double)c; }
  __device__ bool gt_is(int i, int c) const { return (double)gt[5 * (size_t)i + 4] == (double)c; }
  __device__ void pr_box(int i, double& x1, double& y1, double& x2, double& y2) const {
    const float* b = pr + 6 * (size_t)i; x1 = b[0]; y1 = b[1]; x2 = b[2]; y2 = b[3];
  }
  __device__ void gt_box(int i, double& x1, double& y1, double& x2, double& y2) const {
    const float* b = gt + 5 * (size_t)i; x1 = b[0]; y1 = b[1]; x2 = b[2]; y2 = b[3];
  }
  __device__ float pr_score(int i) const { return pr[6 * (size_t)i + 5]; }
};

__global__ void __launch_bounds__(MAP_THREADS) map_kernel(MapParams p) {
  extern __shared__ __align__(16) unsigned char map_smem[];
  const int img = blockIdx.x;
  const int g0 = p.gt_off[img], ng_all = p.gt_off[img + 1] - g0;
  const int p0 = p.pr_off[img], np_all = p.pr_off[img + 1] - p0;
  MapRowsSrc s;
  s.gt = p.gt + 5 * (size_t)g0;
  s.pr = p.pr + 6 * (size_t)p0;
  const double v = map_image(s, np_all, ng_all, p.cap_g, p.class_num, p.thresh, map_smem_carve(map_smem, p.cap_p, p.cap_g));
  if (threadIdx.x == 0) p.out[img] = v;
}

// ---- padded NMS output + ground-truth box lists ----------------------------------------------------------------------
struct MapPaddedParams {
  const float* pr_boxes; const void* pr_cls; const float* pr_scores; const int32_t* pr_count;   // [B,K,4] [B,K] [B,K] [B]
  int K;
  const float* gt_boxes; const int32_t* gt_cls; const int32_t* gt_off; const int32_t* gt_count;  // [total,4] [total] [B+1] [B]|null
  int total_gt;
  int class_num; double thresh;
  double* out;
};

template <typename CI>
struct MapPaddedSrc {
  const float* pb; const CI* pc; const float* ps;   // the image's K prediction slots
  const float* gb; const int32_t* gc;               // the image's ground-truth rows
  __device__ bool pr_is(int i, int c) const { return pc[i] == (CI)c; }
  __device__ bool gt_is(int i, int c) const { return gc[i] == c; }
  __device__ void pr_box(int i, double& x1, double& y1, double& x2, double& y2) const {
    const float* b = pb + 4 * (size_t)i; x1 = b[0]; y1 = b[1]; x2 = b[2]; y2 = b[3];
  }
  __device__ void gt_box(int i, double& x1, double& y1, double& x2, double& y2) const {
    const float* b = gb + 4 * (size_t)i; x1 = b[0]; y1 = b[1]; x2 = b[2]; y2 = b[3];
  }
  __device__ float pr_score(int i) const { return ps[i]; }
};

template <typename CI>
__global__ void __launch_bounds__(MAP_THREADS) map_padded_kernel(MapPaddedParams p) {
  extern __shared__ __align__(16) unsigned char map_smem[];
  const int img = blockIdx.x;
  const size_t pbase = (size_t)img * p.K;
  const int np_all = min(max(p.pr_count[img], 0), p.K);
  // offsets clamped to the ground-truth list: a bad offset cannot reach past it
  const int g0 = min(max(p.gt_off[img], 0), p.total_gt), g_span = max(min(p.gt_off[img + 1], p.total_gt) - g0, 0);
  const int ng_all = p.gt_count ? min(max(p.gt_count[img], 0), g_span) : g_span;
  MapPaddedSrc<CI> s;
  s.pb = p.pr_boxes + 4 * pbase; s.pc = static_cast<const CI*>(p.pr_cls) + pbase; s.ps = p.pr_scores + pbase;
  s.gb = p.gt_boxes + 4 * (size_t)g0; s.gc = p.gt_cls + g0;
  const double v = map_image(s, np_all, ng_all, MAP_GT_CHUNK, p.class_num, p.thresh, map_smem_carve(map_smem, p.K, MAP_GT_CHUNK));
  if (threadIdx.x == 0) p.out[img] = v;
}

extern "C" int b200_map_per_image(const float* gt, const int32_t* gt_offsets, const float* pred,
                                  const int32_t* pred_offsets, int num_images, int max_gt_per_image,
                                  int max_pred_per_image, int class_num, double thresh, double* out, void* stream) {
  B200_REQUIRE(num_images >= 0 && class_num >= 1 && max_gt_per_image >= 0 && max_pred_per_image >= 0, B200_ERR_BAD_ARG,
               "b200_map_per_image: bad sizes");
  if (num_images == 0) return B200_OK;
  B200_REQUIRE(gt_offsets && pred_offsets && out, B200_ERR_BAD_ARG, "b200_map_per_image: null pointer");
  MapParams p;
  p.gt = gt; p.gt_off = gt_offsets; p.pr = pred; p.pr_off = pred_offsets; p.class_num = class_num; p.thresh = thresh;
  p.cap_p = max_pred_per_image > 0 ? max_pred_per_image : 1;
  p.cap_g = max_gt_per_image > 0 ? max_gt_per_image : 1;
  p.out = out;
  const size_t smem = map_smem_bytes(p.cap_p, p.cap_g);
  B200_REQUIRE(smem <= 200 * 1024, B200_ERR_UNSUPPORTED, "b200_map_per_image: too many boxes per image (%d predictions, %d ground truth)",
               max_pred_per_image, max_gt_per_image);
  B200_CUDA(cudaFuncSetAttribute(map_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  map_kernel<<<num_images, MAP_THREADS, smem, (cudaStream_t)stream>>>(p);
  B200_LAUNCH_CHECK();
  return B200_OK;
}

extern "C" int b200_map_padded(const float* pred_boxes, const void* pred_classes, int class_id_bytes, const float* pred_scores,
                               const int32_t* pred_count, int num_images, int max_out, const float* gt_boxes,
                               const int32_t* gt_classes, int total_gt, const int32_t* gt_offsets, const int32_t* gt_count,
                               int class_num, double thresh, double* out, void* stream) {
  const char* who = "b200_map_padded";
  B200_REQUIRE(num_images >= 0, B200_ERR_BAD_ARG, "%s: negative num_images", who);
  B200_REQUIRE(class_num >= 1, B200_ERR_BAD_ARG, "%s: class_num %d < 1", who, class_num);
  B200_REQUIRE(max_out >= 1 && max_out <= NMS_MAX_OUT_LIMIT, B200_ERR_UNSUPPORTED, "%s: max_out %d outside [1,%d]", who, max_out,
               NMS_MAX_OUT_LIMIT);
  B200_REQUIRE(class_id_bytes == 4 || class_id_bytes == 8, B200_ERR_BAD_ARG, "%s: class_id_bytes must be 4 (int32) or 8 (int64), got %d",
               who, class_id_bytes);
  if (num_images == 0) return B200_OK;
  B200_REQUIRE(pred_boxes && pred_classes && pred_scores && pred_count, B200_ERR_BAD_ARG, "%s: null prediction argument", who);
  B200_REQUIRE(gt_offsets && out, B200_ERR_BAD_ARG, "%s: null gt_offsets / out", who);
  B200_REQUIRE(total_gt >= 0, B200_ERR_BAD_ARG, "%s: negative total_gt", who);
  B200_REQUIRE(total_gt == 0 || (gt_boxes && gt_classes), B200_ERR_BAD_ARG, "%s: null gt_boxes / gt_classes", who);
  MapPaddedParams p;
  p.pr_boxes = pred_boxes; p.pr_cls = pred_classes; p.pr_scores = pred_scores; p.pr_count = pred_count; p.K = max_out;
  p.gt_boxes = gt_boxes; p.gt_cls = gt_classes; p.gt_off = gt_offsets; p.gt_count = gt_count; p.total_gt = total_gt;
  p.class_num = class_num; p.thresh = thresh; p.out = out;
  const size_t smem = map_smem_bytes(max_out, MAP_GT_CHUNK);
  cudaStream_t s = (cudaStream_t)stream;
  if (class_id_bytes == 4) {
    B200_CUDA(cudaFuncSetAttribute(map_padded_kernel<int32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    map_padded_kernel<int32_t><<<num_images, MAP_THREADS, smem, s>>>(p);
  } else {
    B200_CUDA(cudaFuncSetAttribute(map_padded_kernel<long long>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    map_padded_kernel<long long><<<num_images, MAP_THREADS, smem, s>>>(p);
  }
  B200_LAUNCH_CHECK();
  return B200_OK;
}
