// Evaluation metrics the reference's drivers compute on the device around the NST path:
//   cal_IoUs (utils.py:163-194; call sites iris_style_transfer_openeds2019.py:156, data_preprocessing.py:168): per image and
//   class the intersection-over-union of two label maps.  The reference makes, per class, two float copies of both maps, a
//   product, a sum, a clamp and two reductions -- ~30 elementwise passes over B x H x W for four classes.  Here ONE pass
//   reads the two maps: for int64 maps (16 B per pixel: HBM-bound) warp ballots turn 32 pixels into one match word per class
//   and map, for uint8 maps (2 B per pixel) each lane counts 16 pixels per 16-byte load inside its registers; popc(p & t) /
//   popc(p | t) count intersection and union exactly either way, and the ratios are formed in fp32 like the reference (the
//   float sums of 0/1 values are exact integers below 2^24, so the results are bit-identical).
//   angular_distance (utils.py:216-240; gaze_estimation.py:85,102,119): acos of the clamped row dot product, and degrees.
#include <algorithm>

#include "../../include/isx.h"
#include "isx_common.cuh"

namespace isx {
namespace {

inline cudaStream_t S(isx_stream s) { return static_cast<cudaStream_t>(s); }
constexpr int kIouThreads = 256;
constexpr int kIouMaxClass = 8;

template <int NC>
__global__ void __launch_bounds__(kIouThreads)
seg_iou_count_kernel(const long long* __restrict__ preds, const long long* __restrict__ targets, long long hw,
                     unsigned int* __restrict__ counts /* [B][NC][2] */) {
  const int b = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const long long warps = static_cast<long long>(gridDim.x) * (kIouThreads / 32);
  const long long* p = preds + static_cast<long long>(b) * hw;
  const long long* t = targets + static_cast<long long>(b) * hw;
  unsigned inter[NC], uni[NC];   // warp-uniform: every lane holds the same counts
#pragma unroll
  for (int c = 0; c < NC; ++c) { inter[c] = 0; uni[c] = 0; }
  constexpr int U = 4;           // 32-pixel groups in flight per warp: 2 x 4 x 256 B
  const long long groups = (hw + 31) / 32;
  for (long long g0 = (static_cast<long long>(blockIdx.x) * (kIouThreads / 32) + (threadIdx.x >> 5)) * U; g0 < groups; g0 += warps * U) {
    long long pv[U], tv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long i = (g0 + u) * 32 + lane;
      const bool in = i < hw;
      pv[u] = in ? p[i] : -1;    // -1 matches no class 0..NC-1
      tv[u] = in ? t[i] : -1;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        const unsigned pm = __ballot_sync(0xffffffffu, pv[u] == c), tm = __ballot_sync(0xffffffffu, tv[u] == c);
        inter[c] += __popc(pm & tm);
        uni[c] += __popc(pm | tm);
      }
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      if (inter[c]) atomicAdd(&counts[(b * NC + c) * 2 + 0], inter[c]);
      if (uni[c]) atomicAdd(&counts[(b * NC + c) * 2 + 1], uni[c]);
    }
  }
}

// 0x80 in every byte of x that is zero, 0 elsewhere; exact (no borrow between bytes, unlike (x - 0x01..) & ~x)
__device__ __forceinline__ unsigned zero_byte_marks(unsigned x) {
  return ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x | 0x7F7F7F7Fu);
}

// The uint8 counterpart of seg_iou_count_kernel.  At 2 B per pixel ballots over 1-byte loads would be issue-bound long before
// HBM, so each lane counts 16 pixels per map from one 16-byte load inside its registers: per class, exact per-byte equality
// marks (bit 7 of each byte) of the four words of each map, the four AND / OR words folded into one by shifting word j
// right by j, one popc each.  Per-lane counts, one warp reduction and one atomic per warp and class at the end.  The bytes
// before the first 16-byte boundary of an image and after the last one (and everything when the two maps are not equally
// aligned) are counted one pixel per thread.
template <int NC>
__global__ void __launch_bounds__(kIouThreads)
seg_iou_count_u8_kernel(const uint8_t* __restrict__ preds, const uint8_t* __restrict__ targets, long long hw,
                        unsigned int* __restrict__ counts /* [B][NC][2] */) {
  const int b = blockIdx.y;
  const long long nthr = static_cast<long long>(gridDim.x) * kIouThreads;
  const long long gt = static_cast<long long>(blockIdx.x) * kIouThreads + threadIdx.x;
  const uint8_t* p = preds + static_cast<long long>(b) * hw;
  const uint8_t* t = targets + static_cast<long long>(b) * hw;
  unsigned inter[NC], uni[NC];   // per lane
#pragma unroll
  for (int c = 0; c < NC; ++c) { inter[c] = 0; uni[c] = 0; }
  const uintptr_t ap = reinterpret_cast<uintptr_t>(p), at = reinterpret_cast<uintptr_t>(t);
  const long long head = ((ap ^ at) & 15) ? hw : std::min<long long>(hw, static_cast<long long>((16 - (ap & 15)) & 15));
  const long long nvec = (hw - head) >> 4, tail = head + nvec * 16;
  auto scalar = [&](long long i) {
    const int pv = p[i], tv = t[i];
#pragma unroll
    for (int c = 0; c < NC; ++c) { inter[c] += (pv == c) & (tv == c); uni[c] += (pv == c) | (tv == c); }
  };
  for (long long i = gt; i < head; i += nthr) scalar(i);
  for (long long i = tail + gt; i < hw; i += nthr) scalar(i);
  const uint4* pv4 = reinterpret_cast<const uint4*>(p + head);
  const uint4* tv4 = reinterpret_cast<const uint4*>(t + head);
  constexpr int U = 2;           // 16-byte loads in flight per lane and map
  for (long long v0 = gt; v0 < nvec; v0 += nthr * U) {
    uint4 pw[U], tw[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long v = v0 + u * nthr;
      pw[u] = v < nvec ? __ldg(pv4 + v) : make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);   // 255: no class
      tw[u] = v < nvec ? __ldg(tv4 + v) : make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        const unsigned k = 0x01010101u * c;
        const unsigned p0 = zero_byte_marks(pw[u].x ^ k), p1 = zero_byte_marks(pw[u].y ^ k);
        const unsigned p2 = zero_byte_marks(pw[u].z ^ k), p3 = zero_byte_marks(pw[u].w ^ k);
        const unsigned t0 = zero_byte_marks(tw[u].x ^ k), t1 = zero_byte_marks(tw[u].y ^ k);
        const unsigned t2 = zero_byte_marks(tw[u].z ^ k), t3 = zero_byte_marks(tw[u].w ^ k);
        inter[c] += __popc((p0 & t0) | ((p1 & t1) >> 1) | ((p2 & t2) >> 2) | ((p3 & t3) >> 3));
        uni[c] += __popc((p0 | t0) | ((p1 | t1) >> 1) | ((p2 | t2) >> 2) | ((p3 | t3) >> 3));
      }
    }
  }
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const unsigned i = __reduce_add_sync(0xffffffffu, inter[c]), u = __reduce_add_sync(0xffffffffu, uni[c]);
    if ((threadIdx.x & 31) == 0) {
      if (i) atomicAdd(&counts[(b * NC + c) * 2 + 0], i);
      if (u) atomicAdd(&counts[(b * NC + c) * 2 + 1], u);
    }
  }
}

// one grid for either map dtype: seg_dtype 0 = int64 (ballots), 1 = uint8 (in-register byte counting)
template <int NC>
void launch_iou_count(int seg_dtype, dim3 grid, cudaStream_t s, const void* p, const void* t, long long hw, unsigned* counts) {
  if (seg_dtype == 1)
    seg_iou_count_u8_kernel<NC><<<grid, kIouThreads, 0, s>>>(static_cast<const uint8_t*>(p), static_cast<const uint8_t*>(t), hw, counts);
  else
    seg_iou_count_kernel<NC><<<grid, kIouThreads, 0, s>>>(static_cast<const long long*>(p), static_cast<const long long*>(t), hw, counts);
}

__global__ void seg_iou_finalize_kernel(const unsigned int* __restrict__ counts, int B, int NC, float eps, float* __restrict__ iou,
                                        float* __restrict__ miou) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float sum = 0.f;
  for (int c = 0; c < NC; ++c) {
    const float i = static_cast<float>(counts[(b * NC + c) * 2 + 0]), u = static_cast<float>(counts[(b * NC + c) * 2 + 1]);
    const float v = __fdiv_rn(i, __fadd_rn(u, eps));   // intersection / (union + eps), utils.py:189
    iou[b * NC + c] = v;
    sum = __fadd_rn(sum, v);
  }
  miou[b] = __fdiv_rn(sum, static_cast<float>(NC));      // ious.mean(dim = 1)
}

__global__ void angular_distance_kernel(const float* __restrict__ v1, const float* __restrict__ v2, int n, int d,
                                        float* __restrict__ radian, float* __restrict__ degree) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float dot = 0.f;
  for (int k = 0; k < d; ++k) dot = __fadd_rn(dot, __fmul_rn(v1[i * d + k], v2[i * d + k]));   // torch.sum(v1 * v2, dim = 1)
  dot = fminf(fmaxf(dot, -1.0f), 1.0f);
  const float r = acosf(dot);
  radian[i] = r;
  degree[i] = r * 57.29577951308232f;   // torch.rad2deg: x * (180 / pi)
}

}  // namespace
}  // namespace isx

using namespace isx;

extern "C" int isx_seg_iou_typed(const void* preds, const void* targets, int seg_dtype, int B, int64_t HW, int num_class,
                                 float eps, uint32_t* counts, float* iou, float* miou, isx_stream stream) {
  ISX_REQUIRE(seg_dtype == 0 || seg_dtype == 1, "isx_seg_iou: seg_dtype %d (0 = int64, 1 = uint8)", seg_dtype);
  ISX_REQUIRE(preds && targets && counts && iou && miou, "isx_seg_iou: null pointer");
  ISX_REQUIRE(B > 0 && B <= 65535 && HW > 0 && HW < (1ll << 32), "isx_seg_iou: bad shape B=%d (1..65535) HW=%lld", B, static_cast<long long>(HW));
  ISX_REQUIRE(num_class >= 1 && num_class <= kIouMaxClass, "isx_seg_iou: num_class %d (1..%d)", num_class, kIouMaxClass);
  cudaStream_t s = S(stream);
  ISX_CHECK_CUDA(cudaMemsetAsync(counts, 0, static_cast<size_t>(B) * num_class * 2 * sizeof(uint32_t), s));
  // two resident waves over the batch (ncu: 768 blocks at 4 resident per SM = 1.3 waves ran at 4.4 TB/s)
  int per_sm = 4;
  long long blocks_needed;   // blocks that give every thread at least one full step of its loop
  if (seg_dtype == 1) {
    ISX_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, seg_iou_count_u8_kernel<4>, kIouThreads, 0));
    blocks_needed = (HW / 16 + kIouThreads * 2 - 1) / (kIouThreads * 2);
  } else {
    ISX_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, seg_iou_count_kernel<4>, kIouThreads, 0));
    const long long groups = (HW + 31) / 32;
    blocks_needed = (groups + 8 * 4 - 1) / (8 * 4);
  }
  const int cap = std::max(1, isx_num_sms() * std::max(1, per_sm) * 2 / B);
  const int bx = static_cast<int>(std::max<long long>(1, std::min<long long>(cap, blocks_needed)));
  const dim3 grid(bx, B);
  switch (num_class) {
    case 1: launch_iou_count<1>(seg_dtype, grid, s, preds, targets, HW, counts); break;
    case 2: launch_iou_count<2>(seg_dtype, grid, s, preds, targets, HW, counts); break;
    case 3: launch_iou_count<3>(seg_dtype, grid, s, preds, targets, HW, counts); break;
    case 4: launch_iou_count<4>(seg_dtype, grid, s, preds, targets, HW, counts); break;
    case 5: launch_iou_count<5>(seg_dtype, grid, s, preds, targets, HW, counts); break;
    case 6: launch_iou_count<6>(seg_dtype, grid, s, preds, targets, HW, counts); break;
    case 7: launch_iou_count<7>(seg_dtype, grid, s, preds, targets, HW, counts); break;
    default: launch_iou_count<8>(seg_dtype, grid, s, preds, targets, HW, counts); break;
  }
  ISX_LAUNCH_CHECK();
  seg_iou_finalize_kernel<<<(B + 127) / 128, 128, 0, s>>>(counts, B, num_class, eps, iou, miou);
  ISX_LAUNCH_CHECK();
  return 0;
}

extern "C" int isx_seg_iou(const int64_t* preds, const int64_t* targets, int B, int64_t HW, int num_class, float eps,
                           uint32_t* counts, float* iou, float* miou, isx_stream stream) {
  return isx_seg_iou_typed(preds, targets, 0, B, HW, num_class, eps, counts, iou, miou, stream);
}

extern "C" int isx_angular_distance(const float* v1, const float* v2, int n, int d, float* radian, float* degree, isx_stream stream) {
  ISX_REQUIRE(v1 && v2 && radian && degree && n > 0 && d > 0, "isx_angular_distance: bad arguments");
  angular_distance_kernel<<<(n + 255) / 256, 256, 0, S(stream)>>>(v1, v2, n, d, radian, degree);
  ISX_LAUNCH_CHECK();
  return 0;
}
