// Row f4 (SURVEY.md §8f): the downstream evaluator's feature path of models/gaze_estimators/gaze_estimators.py on the device.
//
//   extract_eye_landmarks (gaze_estimators.py:108-178; call sites data_preprocessing.py:412, gaze_estimators.py:49,291) is
//   called ONE label map at a time, each call a `.cpu().numpy()` round trip + cv2.findContours / contourArea / fitEllipse
//   for the pupil and the iris + np.where for the sclera.  Here a batch of label maps takes three launches:
//     lm_planes_kernel    labels (int64 / int32 / uint8) -> one BIT per pixel for the pupil and the iris class (warp ballots)
//                         + the sclera's bounding box = the eye corners.  HBM-bound: 8 B/pixel in, 2 bits/pixel out.
//     lm_contour_kernel   one CTA per (frame, class): the class's bit plane and two mark planes live in shared memory
//                         (3 x 34 KB at 400x640).  All threads find, per row, the first outer-border start OpenCV's scanner
//                         would accept; one warp then walks the starts in raster order, one thread follows each border
//                         (Suzuki-Abe as OpenCV implements it: the marks decide which later starts are external) and keeps
//                         the contour of largest area; then all threads accumulate the normal equations of OpenCV's
//                         two-stage conic fit in double-double arithmetic.
//     lm_finalize_kernel  the 19 landmarks per frame (the derived ones in double like the Python arithmetic).
//   The per-pixel / per-point arithmetic is in landmarks_core.cuh, which the CPU tier compiles with g++ and pins against cv2.
//
//   GazeEstimator1 / GazeEstimator2 heads (gaze_estimators.py:24-32,51-53 / :196-204,221-223; eval mode): in -> hidden ->
//   hidden -> out with ReLU between, then x / ||x||_2: one kernel, fp32 FMA (19 or 2048 inputs, 64 hidden units: far too
//   small for a tensor-core tile; the weights stay in L2, four samples share every weight load).
#include <algorithm>
#include <limits.h>

#include "../../include/isx.h"
#include "isx_common.cuh"
#include "landmarks_core.cuh"

namespace isx {
namespace {

using namespace isx_lm;

inline cudaStream_t S(isx_stream s) { return static_cast<cudaStream_t>(s); }
inline size_t lm_align(size_t n) { return (n + 255) & ~static_cast<size_t>(255); }

constexpr int kLmThreads = 256;          // plane kernel
constexpr int kLmContourThreads = 128;   // contour kernel: 228 registers per thread (the double-double fit) -> 128 threads so
                                         // that two CTAs fit on an SM (ncu: 256 threads = one CTA per SM, 1.7 waves for 256 CTAs)

struct LmResult {   // per (frame, class)
  float box[5];     // cx, cy, width, height, angle
  int n_points;     // points of the chosen contour
  int n_contours;   // external contours found
  int flags;        // 1: five points or rank-deficient system (OpenCV leaves the general algorithm there), 2: more than max_points
  int has;          // an ellipse was fitted
};

__global__ void lm_init_kernel(int32_t* sclera, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) { sclera[b * 4 + 0] = INT_MAX; sclera[b * 4 + 1] = -1; sclera[b * 4 + 2] = INT_MAX; sclera[b * 4 + 3] = -1; }
}

// planes[b][cls][y][w]: bit x & 31 of word x >> 5 is (uint8)label == (cls == 0 ? 3 : 2); sclera[b] = {xmin, xmax, ymin, ymax}.
// A warp owns whole rows: lane l reads pixel 32 w + l of word w (one 256-byte request per warp and word, U requests in
// flight), three ballots turn the 32 labels into the bits of the pupil / iris word and into the sclera's column range -- the
// ballots are warp-uniform, so the bounding box needs no reduction.  No division, ~15 instructions per 256 bytes (the first
// version indexed a flat word list: two integer divisions per word, 52 instructions, 67 % of the issue slots, 3.1 TB/s).
template <typename T, int U>
__global__ void __launch_bounds__(kLmThreads)
lm_planes_kernel(const T* __restrict__ seg, uint32_t* __restrict__ planes, int32_t* __restrict__ sclera, int H, int W, int Wu) {
  const int b = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int warps = gridDim.x * (kLmThreads / 32);
  const T* img = seg + static_cast<size_t>(b) * H * W;
  uint32_t* p3 = planes + static_cast<size_t>(b) * 2 * H * Wu;
  uint32_t* p2 = p3 + static_cast<size_t>(H) * Wu;
  int xmin = INT_MAX, xmax = -1, ymin = INT_MAX, ymax = -1;
  for (int y = blockIdx.x * (kLmThreads / 32) + (threadIdx.x >> 5); y < H; y += warps) {
    const T* row = img + static_cast<size_t>(y) * W;
    bool any = false;
    for (int w0 = 0; w0 < Wu; w0 += U) {
      unsigned v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int x = (w0 + u) * 32 + lane;
        v[u] = x < W ? (static_cast<unsigned>(row[x]) & 255u) : 0u;   // astype(np.uint8); words past the row read as background
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const unsigned b3 = __ballot_sync(0xffffffffu, v[u] == 3u), b2 = __ballot_sync(0xffffffffu, v[u] == 2u);
        const unsigned b1 = __ballot_sync(0xffffffffu, v[u] == 1u);
        if (w0 + u < Wu && lane == 0) { p3[y * Wu + w0 + u] = b3; p2[y * Wu + w0 + u] = b2; }
        if (b1) {
          xmin = min(xmin, (w0 + u) * 32 + __ffs(static_cast<int>(b1)) - 1);
          xmax = max(xmax, (w0 + u) * 32 + 31 - __clz(static_cast<int>(b1)));
          any = true;
        }
      }
    }
    if (any) { ymin = min(ymin, y); ymax = y; }   // rows ascend
  }
  if (lane == 0 && xmax >= 0) {
    atomicMin(&sclera[b * 4 + 0], xmin); atomicMax(&sclera[b * 4 + 1], xmax);
    atomicMin(&sclera[b * 4 + 2], ymin); atomicMax(&sclera[b * 4 + 3], ymax);
  }
}

// lm_row_first_start (landmarks_core.cuh) for ONE row by a whole warp, Ww <= 32: lane w owns word w.  The two things the
// serial scan carries from word to word -- the foreground bit left of the word and the sign of the last marked pixel so far --
// come from a shuffle and from two ballots, so a row costs ~50 instructions instead of ~12 per word in sequence.  Used for
// the rescan after a contour of a few rows (every stray speck: 1.8 -> 0.6 us per stray contour); all 32 lanes must call it.
__device__ __forceinline__ int lm_row_first_start_warp(const uint32_t* F, const uint32_t* M, const uint32_t* N, int Ww, int y,
                                                       int x_after, int lane) {
  const bool own = lane < Ww;
  const uint32_t fw = own ? F[y * Ww + lane] : 0u;
  const uint32_t mw = fw ? M[y * Ww + lane] : 0u, nw = fw ? N[y * Ww + lane] : 0u;   // marks exist on foreground only
  uint32_t prev_top = __shfl_up_sync(0xffffffffu, fw >> 31, 1);
  if (lane == 0) prev_top = 0u;
  const uint32_t cand = lm_word_candidates(fw, mw, prev_top, x_after, lane);
  const unsigned bal_has = __ballot_sync(0xffffffffu, mw != 0u), bal_pos = __ballot_sync(0xffffffffu, lm_word_last_mark_positive(mw, nw));
  const unsigned below = bal_has & ((1u << lane) - 1u);   // words left of this one that carry a mark
  const int inside_in = below ? static_cast<int>((bal_pos >> (31 - __clz(static_cast<int>(below)))) & 1u) : 0;
  const int k = lm_word_first_accepted(cand, mw, nw, inside_in);
  const int x = k >= 0 ? lane * 32 + k : -1;
  const unsigned found = __ballot_sync(0xffffffffu, x >= 0);
  if (!found) return -1;
  return __shfl_sync(0xffffffffu, x, __ffs(static_cast<int>(found)) - 1);
}

// sum of K doubles per thread over the block; the totals are returned to every thread in v[]
template <int K>
__device__ void lm_block_sum(double* v, double* red /* [kLmContourThreads / 32][K] shared */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    double x = v[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0) red[warp * K + k] = x;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < K; ++k) {
    double x = 0;
#pragma unroll
    for (int w = 0; w < kLmContourThreads / 32; ++w) x += red[w * K + k];
    v[k] = x;
  }
  __syncthreads();
}

// the same for double-double accumulators
template <int K>
__device__ void lm_block_sum_dd(dd* v, dd* red /* [kLmContourThreads / 32][K] shared */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    dd x = v[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      dd y;
      y.hi = __shfl_xor_sync(0xffffffffu, x.hi, o);
      y.lo = __shfl_xor_sync(0xffffffffu, x.lo, o);
      x = dd_add(x, y);
    }
    if (lane == 0) red[warp * K + k] = x;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < K; ++k) {
    dd x = red[k];
#pragma unroll
    for (int w = 1; w < kLmContourThreads / 32; ++w) x = dd_add(x, red[w * K + k]);
    v[k] = x;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kLmContourThreads, 2)
lm_contour_kernel(const uint32_t* __restrict__ planes, uint32_t* __restrict__ points, LmResult* __restrict__ results, int H, int W,
                  int Wu, int Ww, int cap) {
  extern __shared__ uint32_t lm_smem[];
  const int cls = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const int rows = H + 2, pw = rows * Ww;
  uint32_t* F = lm_smem;
  uint32_t* M = F + pw;
  uint32_t* N = M + pw;
  __shared__ int s_best_n, s_best_buf, s_ncont;
  __shared__ dd s_red_dd[(kLmContourThreads / 32) * kLmSums1];
  double* s_red = reinterpret_cast<double*>(s_red_dd);
  __shared__ double s_bcast[8];

  // ---- the class's bit plane with its one-pixel zero frame: bit (x + 1) of row (y + 1) ----
  const uint32_t* G = planes + (static_cast<size_t>(b) * 2 + cls) * H * Wu;
  for (int i = tid; i < pw; i += kLmContourThreads) {
    const int yp = i / Ww, w = i - yp * Ww;
    uint32_t f = 0;
    if (yp >= 1 && yp <= H) {
      const uint32_t* g = G + (yp - 1) * Wu;
      const uint32_t lo = w < Wu ? g[w] : 0u, hi = (w >= 1 && w - 1 < Wu) ? g[w - 1] : 0u;
      f = (lo << 1) | (hi >> 31);
    }
    F[i] = f; M[i] = 0u; N[i] = 0u;
  }
  __syncthreads();

  // ---- raster scan + border following, contour by contour in OpenCV's order of discovery ----
  // cand[y] = first start OpenCV's scanner would accept in padded row y (-1: none).  All threads fill it once; then ONE WARP
  // runs the sequential part without block barriers: find the first row with a candidate (ballots), lane 0 follows that
  // border, and only the rows the trace touched (start row .. y_max: a trace marks nothing else, rows above the start are
  // done) are rescanned, one row per lane.
  int* cand = reinterpret_cast<int*>(N + pw);
  for (int y = tid; y < rows; y += kLmContourThreads) cand[y] = (y >= 1 && y <= H) ? lm_row_first_start(F, M, N, Ww, y, 0) : -1;
  __syncthreads();
  uint32_t* buf0 = points + (static_cast<size_t>(b) * 2 + cls) * 2 * cap;
  if (tid < 32) {
    const int lane = tid;
    long long best_area = -1;
    int best_n = 0, best_buf = 0, cur_buf = 0, ncont = 0, sy = 1;
    for (;;) {
      int fy = -1;
      for (int base = sy; base <= H; base += 32) {
        const int y = base + lane;
        const unsigned bal = __ballot_sync(0xffffffffu, y <= H && cand[y] >= 0);
        if (bal) { fy = base + __ffs(static_cast<int>(bal)) - 1; break; }
      }
      if (fy < 0) break;
      const int x0 = cand[fy];
      int y_max = fy;
      if (lane == 0) {
        const LmTrace t = lm_trace(F, M, N, Ww, x0, fy, buf0 + static_cast<size_t>(cur_buf) * cap, cap);
        const long long a = t.cross < 0 ? -t.cross : t.cross;
        if (a >= best_area) {   // cv2 returns the contours in reverse order of discovery and max() keeps the first maximum
          best_area = a; best_n = t.n; best_buf = cur_buf; cur_buf ^= 1;
        }
        ++ncont;
        y_max = t.y_max;
      }
      y_max = __shfl_sync(0xffffffffu, y_max, 0);   // also orders lane 0's mark writes before the rescans
      __syncwarp();
      if (y_max - fy < 6 && Ww <= 32) {   // a stray speck (a few rows at most): warp-wide rescans, row after row
        for (int y = fy; y <= y_max; ++y) {
          const int x = lm_row_first_start_warp(F, M, N, Ww, y, y == fy ? x0 : 0, lane);
          if (lane == 0) cand[y] = x;
        }
      } else {
        for (int y = fy + lane; y <= y_max; y += 32) cand[y] = lm_row_first_start(F, M, N, Ww, y, y == fy ? x0 : 0);
      }
      __syncwarp();
      sy = fy;
    }
    if (lane == 0) { s_best_n = best_n; s_best_buf = best_buf; s_ncont = ncont; }
  }
  __syncthreads();

  // ---- cv2.fitEllipse of the chosen contour ----
  const int n = s_best_n;
  LmResult* res = results + b * 2 + cls;
  int flags = 0, has = 0;
  float box[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
  if (n > cap) {
    flags |= 2;
  } else if (n >= 5) {
    __threadfence_block();
    const uint32_t* pts = buf0 + static_cast<size_t>(s_best_buf) * cap;   // written by thread 0 of this block
    double v[2];
    v[0] = 0; v[1] = 0;
    for (int i = tid; i < n; i += kLmContourThreads) { const uint32_t p = pts[i]; v[0] += p & 0xFFFFu; v[1] += p >> 16; }
    lm_block_sum<2>(v, s_red);
    // Point2f c += p; c /= n  (integer-valued float sums below 2^24 are exact in any order)
    const float cx = __fdiv_rn(static_cast<float>(v[0]), static_cast<float>(n)), cy = __fdiv_rn(static_cast<float>(v[1]), static_cast<float>(n));
    v[0] = 0;
    for (int i = tid; i < n; i += kLmContourThreads) {
      const uint32_t p = pts[i];
      const float dx = __fsub_rn(static_cast<float>(p & 0xFFFFu), cx), dy = __fsub_rn(static_cast<float>(p >> 16), cy);
      v[0] += static_cast<double>(__fadd_rn(fabsf(dx), fabsf(dy)));
    }
    lm_block_sum<1>(v, s_red);
    const double scale = 100.0 / (v[0] > 1.1920928955078125e-07 ? v[0] : 1.1920928955078125e-07);
    dd a[kLmSums1];
#pragma unroll
    for (int k = 0; k < kLmSums1; ++k) a[k] = dd_make(0.0);
    for (int i = tid; i < n; i += kLmContourThreads) {
      const uint32_t p = pts[i];
      const float dx = __fsub_rn(static_cast<float>(p & 0xFFFFu), cx), dy = __fsub_rn(static_cast<float>(p >> 16), cy);
      lm_acc1(dx * scale, dy * scale, a);
    }
    lm_block_sum_dd<kLmSums1>(a, s_red_dd);
    if (tid == 0) {
      double gfp[5], rx = 0, ry = 0;
      double piv = 1.0, det = 0.0;
      const bool ok = lm_solve_sym<5>(a, a + 15, gfp, &piv, &det) && lm_centre(gfp, &rx, &ry);
      const int f = (n == 5 || piv < kLmPivotFloor || (!lm_rank_surely_full(a, det) && lm_rank_deficient(a))) ? 1 : 0;
      s_bcast[0] = rx; s_bcast[1] = ry; s_bcast[2] = ok ? 1.0 : 0.0; s_bcast[3] = f;
    }
    __syncthreads();
    const double rx = s_bcast[0], ry = s_bcast[1];
    const bool ok1 = s_bcast[2] != 0.0;
    flags |= static_cast<int>(s_bcast[3]);
#pragma unroll
    for (int k = 0; k < kLmSums2; ++k) a[k] = dd_make(0.0);
    if (ok1) {
      for (int i = tid; i < n; i += kLmContourThreads) {
        const uint32_t p = pts[i];
        const float dx = __fsub_rn(static_cast<float>(p & 0xFFFFu), cx), dy = __fsub_rn(static_cast<float>(p >> 16), cy);
        lm_acc2(dx * scale, dy * scale, rx, ry, a);
      }
    }
    lm_block_sum_dd<kLmSums2>(a, s_red_dd);
    if (tid == 0) {
      double g[3], piv = 1.0;
      if (ok1 && lm_solve_sym<3>(a, a + 6, g, &piv)) lm_box(g, rx, ry, scale, cx, cy, box);
      if (piv < kLmPivotFloor) flags |= 1;   // (numerically) singular: whatever stands in box is not OpenCV's answer
      has = 1;
    }
  }
  if (tid == 0) {
#pragma unroll
    for (int i = 0; i < 5; ++i) res->box[i] = box[i];
    res->n_points = n; res->n_contours = s_ncont; res->flags = flags; res->has = has;
  }
}

__global__ void lm_finalize_kernel(const LmResult* __restrict__ results, const int32_t* __restrict__ sclera, double epsilon,
                                   float* __restrict__ out, int32_t* __restrict__ info, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const LmResult p = results[b * 2 + 0], q = results[b * 2 + 1];
  const int bb[4] = {sclera[b * 4 + 0], sclera[b * 4 + 1], sclera[b * 4 + 2], sclera[b * 4 + 3]};
  float lm[19];
  lm_assemble(p.box, p.has, q.box, q.has, bb, bb[1] >= 0, epsilon, lm);
  for (int i = 0; i < 19; ++i) out[b * 19 + i] = lm[i];
  if (info) {
    int32_t* o = info + b * 8;
    o[0] = p.n_points; o[1] = p.n_contours; o[2] = p.flags; o[3] = q.n_points; o[4] = q.n_contours; o[5] = q.flags;
    o[6] = bb[1] >= 0; o[7] = 0;
  }
}

// ---- gaze heads ----
constexpr int kGhSamples = 4;   // samples per warp: every weight load feeds four accumulators
constexpr int kGhWarps = 4;

// y[s][j] = act(b[j] + sum_k W[j][k] x[s][k]) for the warp's samples; lanes stride over k (coalesced weight rows)
__device__ __forceinline__ void gh_dense(const float* __restrict__ W, const float* __restrict__ bias, int K, int Nout, bool relu,
                                         const float* x /* shared [kGhSamples][K] */, float* y /* shared [kGhSamples][Nout] */) {
  const int lane = threadIdx.x & 31;
  for (int j = 0; j < Nout; ++j) {
    const float* w = W + static_cast<size_t>(j) * K;
    float acc[kGhSamples];
#pragma unroll
    for (int s = 0; s < kGhSamples; ++s) acc[s] = 0.f;
    for (int k = lane; k < K; k += 32) {
      const float wv = __ldg(w + k);
#pragma unroll
      for (int s = 0; s < kGhSamples; ++s) acc[s] = fmaf(wv, x[s * K + k], acc[s]);
    }
#pragma unroll
    for (int s = 0; s < kGhSamples; ++s) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc[s] += __shfl_xor_sync(0xffffffffu, acc[s], o);
    }
    if (lane == 0) {
      const float bj = bias[j];
#pragma unroll
      for (int s = 0; s < kGhSamples; ++s) {
        const float v = acc[s] + bj;
        y[s * Nout + j] = relu ? fmaxf(v, 0.f) : v;
      }
    }
  }
  __syncwarp();
}

__global__ void __launch_bounds__(kGhWarps * 32)
gaze_head_kernel(const float* __restrict__ x, int64_t ldx, int B, int K, int Hd, int O, const float* __restrict__ W1,
                 const float* __restrict__ b1, const float* __restrict__ W2, const float* __restrict__ b2,
                 const float* __restrict__ W3, const float* __restrict__ b3, float* __restrict__ out) {
  extern __shared__ float gh_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int per_warp = kGhSamples * (K + 2 * Hd + O);
  float* xs = gh_smem + warp * per_warp;
  float* h1 = xs + kGhSamples * K;
  float* h2 = h1 + kGhSamples * Hd;
  float* o = h2 + kGhSamples * Hd;
  const int s0 = (blockIdx.x * kGhWarps + warp) * kGhSamples;
  if (s0 >= B) return;
  for (int s = 0; s < kGhSamples; ++s) {
    const int r = min(s0 + s, B - 1);   // the tail repeats the last sample; only rows < B are stored
    for (int k = lane; k < K; k += 32) xs[s * K + k] = x[static_cast<size_t>(r) * ldx + k];
  }
  __syncwarp();
  gh_dense(W1, b1, K, Hd, true, xs, h1);
  gh_dense(W2, b2, Hd, Hd, true, h1, h2);
  gh_dense(W3, b3, Hd, O, false, h2, o);
  if (lane < kGhSamples && s0 + lane < B) {
    float ss = 0.f;
    for (int j = 0; j < O; ++j) ss = fmaf(o[lane * O + j], o[lane * O + j], ss);
    const float nrm = sqrtf(ss);
    for (int j = 0; j < O; ++j) out[static_cast<size_t>(s0 + lane) * O + j] = o[lane * O + j] / nrm;   // x / torch.norm(x, dim=1)
  }
}

struct LmLayout {
  size_t planes, sclera, results, points, total;
  int Wu, Ww;
};
LmLayout lm_layout(int B, int H, int W, int cap) {
  LmLayout L;
  L.Wu = (W + 31) / 32;
  L.Ww = (W + 2 + 31) / 32;
  size_t off = 0;
  L.planes = off; off += lm_align(static_cast<size_t>(B) * 2 * H * L.Wu * 4);
  L.sclera = off; off += lm_align(static_cast<size_t>(B) * 4 * 4);
  L.results = off; off += lm_align(static_cast<size_t>(B) * 2 * sizeof(LmResult));
  L.points = off; off += lm_align(static_cast<size_t>(B) * 2 * 2 * cap * 4);
  L.total = off;
  return L;
}

}  // namespace
}  // namespace isx

using namespace isx;

extern "C" int64_t isx_eye_landmarks_workspace_bytes(int B, int H, int W, int max_points) {
  if (B <= 0 || H <= 0 || W <= 0 || max_points < 5) return -1;
  return static_cast<int64_t>(lm_layout(B, H, W, max_points).total);
}

extern "C" int isx_eye_landmarks(const void* seg, int seg_dtype, int B, int H, int W, double epsilon, int max_points,
                                 void* workspace, float* landmarks, int32_t* info, isx_stream stream) {
  ISX_REQUIRE(seg && workspace && landmarks && B > 0 && H > 0 && W > 0 && max_points >= 5, "isx_eye_landmarks: bad arguments");
  ISX_REQUIRE(seg_dtype >= 0 && seg_dtype <= 2, "isx_eye_landmarks: seg_dtype %d (0 = int64, 1 = uint8, 2 = int32)", seg_dtype);
  ISX_REQUIRE(H < 32768 && W < 65535, "isx_eye_landmarks: frame %dx%d too large for 16-bit point coordinates", H, W);
  ISX_REQUIRE(B <= 65535, "isx_eye_landmarks: at most 65535 label maps per call (got %d)", B);
  const LmLayout L = lm_layout(B, H, W, max_points);
  const size_t smem = static_cast<size_t>(3) * (H + 2) * L.Ww * 4 + static_cast<size_t>(H + 2) * 4;
  ISX_REQUIRE(smem <= 200 * 1024, "isx_eye_landmarks: the three bit planes of a %dx%d frame (%zu bytes) do not fit in shared "
              "memory (the reference asserts 400x640, gaze_estimators.py:121)", H, W, smem);
  cudaStream_t s = S(stream);
  char* ws = static_cast<char*>(workspace);
  uint32_t* planes = reinterpret_cast<uint32_t*>(ws + L.planes);
  int32_t* sclera = reinterpret_cast<int32_t*>(ws + L.sclera);
  LmResult* results = reinterpret_cast<LmResult*>(ws + L.results);
  uint32_t* points = reinterpret_cast<uint32_t*>(ws + L.points);
  lm_init_kernel<<<(B + 127) / 128, 128, 0, s>>>(sclera, B);
  ISX_LAUNCH_CHECK();
  // blocks per frame: TWO resident waves over the batch (measured on a B200, 128 maps: half a wave 3.4 TB/s, one 4.1, one and a
  // half 4.1, two 4.4), at least one block, at most one warp per row.  10 requests in flight per warp (5 / 10 / 20 measured:
  // no difference).
  auto launch = [&](auto kernel, const auto* segp) -> int {
    int per_sm = 1;
    ISX_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kLmThreads, 0));
    const int cap_blocks = std::max(1, isx_num_sms() * std::max(1, per_sm) * 2);
    const int bx = std::max(1, std::min(cap_blocks / B, (H + kLmThreads / 32 - 1) / (kLmThreads / 32)));
    const double label_bytes = seg_dtype == 0 ? 8.0 : seg_dtype == 1 ? 1.0 : 4.0;
    isx_prof_begin(ISX_PROF_PLANES, static_cast<double>(B) * H * (W * label_bytes + 2.0 * L.Wu * 4), s);   // labels in, two bit planes out
    kernel<<<dim3(bx, B), kLmThreads, 0, s>>>(segp, planes, sclera, H, W, L.Wu);
    isx_prof_end(ISX_PROF_PLANES, s);
    ISX_LAUNCH_CHECK();
    return 0;
  };
  int rc = 0;
  if (seg_dtype == 0) {
    rc = launch(lm_planes_kernel<long long, 10>, static_cast<const long long*>(seg));
  } else if (seg_dtype == 1) {
    rc = launch(lm_planes_kernel<uint8_t, 10>, static_cast<const uint8_t*>(seg));
  } else {
    rc = launch(lm_planes_kernel<int, 10>, static_cast<const int*>(seg));
  }
  if (rc) return rc;
  ISX_CHECK_CUDA(cudaFuncSetAttribute(lm_contour_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  ISX_CHECK_CUDA(cudaFuncSetAttribute(lm_contour_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  lm_contour_kernel<<<dim3(2, B), kLmContourThreads, smem, s>>>(planes, points, results, H, W, L.Wu, L.Ww, max_points);
  ISX_LAUNCH_CHECK();
  lm_finalize_kernel<<<(B + 127) / 128, 128, 0, s>>>(results, sclera, epsilon, landmarks, info, B);
  ISX_LAUNCH_CHECK();
  return 0;
}

extern "C" int isx_gaze_head_fwd(const float* x, int64_t ld_x, int B, int in_dim, int hidden, int out_dim, const float* W1,
                                 const float* b1, const float* W2, const float* b2, const float* W3, const float* b3, float* out,
                                 isx_stream stream) {
  ISX_REQUIRE(x && W1 && b1 && W2 && b2 && W3 && b3 && out, "isx_gaze_head_fwd: null pointer");
  ISX_REQUIRE(B > 0 && in_dim > 0 && hidden > 0 && out_dim > 0 && ld_x >= in_dim, "isx_gaze_head_fwd: bad shape");
  const size_t smem = static_cast<size_t>(kGhWarps) * kGhSamples * (in_dim + 2 * hidden + out_dim) * sizeof(float);
  ISX_REQUIRE(smem <= 200 * 1024, "isx_gaze_head_fwd: in_dim %d / hidden %d too large (%zu bytes of shared memory)", in_dim, hidden, smem);
  ISX_CHECK_CUDA(cudaFuncSetAttribute(gaze_head_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const int per_block = kGhWarps * kGhSamples;
  gaze_head_kernel<<<(B + per_block - 1) / per_block, kGhWarps * 32, smem, S(stream)>>>(x, ld_x, B, in_dim, hidden, out_dim, W1, b1, W2, b2,
                                                                                       W3, b3, out);
  ISX_LAUNCH_CHECK();
  return 0;
}
