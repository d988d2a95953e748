// compact.cu — order-preserving row compaction (tf.boolean_mask) and GetGroudTruth.
//
//   tf.boolean_mask in GetBoxes (utils/tf_yolo_utils.py:163-166) and GetGroudTruth (yolo_v4/model.py:380-395)
//   keeps rows in row-major order.  row_positions: flags[n] -> exclusive prefix pos[n] + total, three launches
//   (per-CTA counts, single-CTA scan of the counts, per-CTA ballot prefix); gather_rows copies the flagged rows of
//   a [n, row_floats] array to their positions, one warp per row.
#include "common.cuh"
#include "detmath.h"
#include "yolo_targets.cuh"

#define CP_THREADS 256

__global__ void __launch_bounds__(CP_THREADS) cp_count_kernel(const unsigned char* __restrict__ flags, long long n, int* __restrict__ cta_counts) {
  const long long i = (long long)blockIdx.x * CP_THREADS + threadIdx.x;
  const int f = (i < n && flags[i]) ? 1 : 0;
  const int c = __syncthreads_count(f);
  if (threadIdx.x == 0) cta_counts[blockIdx.x] = c;
}

// exclusive scan of cta_counts[0..m) in place, total -> *total
__global__ void __launch_bounds__(1024) cp_scan_kernel(int* __restrict__ cta_counts, int m, int* __restrict__ total) {
  __shared__ int s_warp[32];
  __shared__ int s_run;
  if (threadIdx.x == 0) s_run = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int base = 0; base < m; base += 1024) {
    const int i = base + threadIdx.x;
    const int v = i < m ? cta_counts[i] : 0;
    int inc = warp_scan_incl(v);
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      const int w = s_warp[lane];
      const int winc = warp_scan_incl(w);
      s_warp[lane] = winc - w;
    }
    __syncthreads();
    const int run = s_run;
    if (i < m) cta_counts[i] = run + s_warp[warp] + inc - v;
    __syncthreads();
    if (threadIdx.x == 1023) s_run = run + s_warp[31] + inc;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = s_run;
}

__global__ void __launch_bounds__(CP_THREADS) cp_positions_kernel(const unsigned char* __restrict__ flags, long long n,
                                                                  const int* __restrict__ cta_offsets, int* __restrict__ pos) {
  __shared__ int s_warp[CP_THREADS / 32];
  const long long i = (long long)blockIdx.x * CP_THREADS + threadIdx.x;
  const bool f = (i < n) && flags[i];
  const uint32_t bal = __ballot_sync(0xffffffffu, f);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) s_warp[warp] = __popc(bal);
  __syncthreads();
  int off = cta_offsets[blockIdx.x];
  for (int w = 0; w < warp; ++w) off += s_warp[w];
  if (i < n) pos[i] = off + __popc(bal & ((1u << lane) - 1u));
}

__global__ void __launch_bounds__(CP_THREADS) cp_gather_rows_kernel(const float* __restrict__ src, int row_floats,
                                                                    const unsigned char* __restrict__ flags,
                                                                    const int* __restrict__ pos, long long n,
                                                                    float* __restrict__ dst) {
  const int lane = threadIdx.x & 31;
  long long row = (long long)blockIdx.x * (CP_THREADS / 32) + (threadIdx.x >> 5);
  const long long stride = (long long)gridDim.x * (CP_THREADS / 32);
  for (; row < n; row += stride) {
    if (!flags[row]) continue;
    const float* s = src + row * row_floats;
    float* d = dst + (long long)pos[row] * row_floats;
    for (int c = lane; c < row_floats; c += 32) d[c] = __ldg(s + c);
  }
}

// GetGroudTruth: per record [x1,y1,x2,y2,class] + flag (conf != 0)
__global__ void __launch_bounds__(CP_THREADS) yolo_ground_truth_rows_kernel(const float* __restrict__ y, long long n, int RF,
                                                                            float* __restrict__ rows,
                                                                            unsigned char* __restrict__ flags) {
  const long long i = (long long)blockIdx.x * CP_THREADS + threadIdx.x;
  if (i >= n) return;
  const float* r = y + i * RF;
  const float conf = __ldg(r + 4);
  const bool f = conf != 0.0f;
  flags[i] = f ? 1 : 0;
  if (!f) return;
  const float x = __ldg(r), yy = __ldg(r + 1), w = __ldg(r + 2), h = __ldg(r + 3);
  int best = 0;
  float bv = __ldg(r + 5);
  for (int c = 1; c < RF - 5; ++c) { const float v = __ldg(r + 5 + c); if (v > bv) { bv = v; best = c; } }  // first max
  float* o = rows + i * 5;
  yolo_gt_corners(x, yy, w, h, o);
  o[4] = (float)best;
}

extern "C" size_t b200_row_positions_workspace_bytes(long long n) {
  const long long m = (n + CP_THREADS - 1) / CP_THREADS;
  return b200_align_up(sizeof(int) * (size_t)(m > 0 ? m : 1), 256);
}

extern "C" int b200_row_positions(const unsigned char* flags, long long n, int* pos, int* total, void* workspace,
                                  size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  B200_REQUIRE(n >= 0 && total, B200_ERR_BAD_ARG, "b200_row_positions: bad argument");
  if (n == 0) { B200_CUDA(cudaMemsetAsync(total, 0, sizeof(int), stream)); return B200_OK; }
  B200_REQUIRE(flags && pos, B200_ERR_BAD_ARG, "b200_row_positions: null pointer");
  const long long m = (n + CP_THREADS - 1) / CP_THREADS;
  B200_REQUIRE(m < (1ll << 31), B200_ERR_UNSUPPORTED, "b200_row_positions: too many rows");
  B200_REQUIRE(workspace && workspace_bytes >= sizeof(int) * (size_t)m, B200_ERR_WORKSPACE, "b200_row_positions: workspace too small");
  int* cta = static_cast<int*>(workspace);
  cp_count_kernel<<<(int)m, CP_THREADS, 0, stream>>>(flags, n, cta);
  B200_LAUNCH_CHECK();
  cp_scan_kernel<<<1, 1024, 0, stream>>>(cta, (int)m, total);
  B200_LAUNCH_CHECK();
  cp_positions_kernel<<<(int)m, CP_THREADS, 0, stream>>>(flags, n, cta, pos);
  B200_LAUNCH_CHECK();
  return B200_OK;
}

extern "C" int b200_gather_rows(const float* src, int row_floats, const unsigned char* flags, const int* pos, long long n,
                                float* dst, void* stream) {
  B200_REQUIRE(n >= 0 && row_floats >= 1, B200_ERR_BAD_ARG, "b200_gather_rows: bad argument");
  if (n == 0) return B200_OK;
  B200_REQUIRE(src && flags && pos && dst, B200_ERR_BAD_ARG, "b200_gather_rows: null pointer");
  long long blocks = (n + 7) / 8;
  const long long cap = (long long)b200_sm_count() * 16;
  if (blocks > cap) blocks = cap;
  cp_gather_rows_kernel<<<(int)blocks, CP_THREADS, 0, (cudaStream_t)stream>>>(src, row_floats, flags, pos, n, dst);
  B200_LAUNCH_CHECK();
  return B200_OK;
}

extern "C" int b200_yolo_ground_truth_rows(const float* y, long long n_records, int C, float* rows, unsigned char* flags,
                                           void* stream) {
  B200_REQUIRE(n_records >= 0 && C >= 1, B200_ERR_BAD_ARG, "b200_yolo_ground_truth_rows: bad argument");
  if (n_records == 0) return B200_OK;
  B200_REQUIRE(y && rows && flags, B200_ERR_BAD_ARG, "b200_yolo_ground_truth_rows: null pointer");
  const long long m = (n_records + CP_THREADS - 1) / CP_THREADS;
  yolo_ground_truth_rows_kernel<<<(int)m, CP_THREADS, 0, (cudaStream_t)stream>>>(y, n_records, 5 + C, rows, flags);
  B200_LAUNCH_CHECK();
  return B200_OK;
}
