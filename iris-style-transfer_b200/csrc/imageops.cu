// K10 / K9: iris mask + bounding box (pipelines.py:139-165, utils.py:44-72) and the composite back
// into the eye frame (iris_style_transfer_openeds2019.py:111-130, …2020.py:121-139), including
// torchvision's antialiased bilinear Resize (ATen _upsample_bilinear2d_aa).  Integer / index work is
// bit-exact; the resize is fp32 with the reference's summation order (W pass inside, H pass outside).
//
// HBM-bound byte work: 128-bit accesses where the row length allows, warp-shuffle bbox reduction, one launch
// per batch with ragged per-image windows; the resize computes the filter taps of a 32x8 output tile ONCE
// into shared memory (they depend on the column / row only) and, in composite mode, does nothing for
// pixels the mask discards.
#include <algorithm>
#include <limits.h>
#include <type_traits>

#include "../../include/isx.h"
#include "isx_common.cuh"

namespace isx {

// bbox[b] = {row_min, col_min, row_max, col_max}; caller-visible sentinel for "no nonzero pixel": row_max = -1
__global__ void bbox_init_kernel(int32_t* bbox, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) {
    bbox[b * 4 + 0] = INT_MAX; bbox[b * 4 + 1] = INT_MAX; bbox[b * 4 + 2] = -1; bbox[b * 4 + 3] = -1;
  }
}

// m = (seg == label) & (x <= thr)   [either test may be disabled]; xm = x * m; bbox over xm != 0.
// T = int64_t or uint8_t label maps; a uint8 label compares as int(seg) == label, so the result equals the int64 path on the
// widened map for every label (one outside 0..255 matches nothing).
// VEC = 4: four pixels per thread (float4 loads, 2 x longlong2 or one uchar4 label load, uchar4 / float4 stores); needs
// W % 4 == 0, 16-byte aligned x / xm and int64 rows, 4-byte aligned uint8 rows, which the launcher checks.
template <int VEC, typename T>
__global__ void __launch_bounds__(256)
mask_bbox_kernel(const float* __restrict__ x, const T* __restrict__ seg, int label, int use_thr, float thr,
                 uint8_t* __restrict__ mask, float* __restrict__ xm, int32_t* __restrict__ bbox, int H, int W) {
  using Lab = typename std::conditional<sizeof(T) == 8, long long, int>::type;
  const int b = blockIdx.y;
  const long hw = static_cast<long>(H) * W;
  const long nv = hw / VEC;
  int rmin = INT_MAX, cmin = INT_MAX, rmax = -1, cmax = -1;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < nv;
       i += static_cast<long>(gridDim.x) * blockDim.x) {
    const long e = i * VEC;
    float v[VEC];
    Lab sg[VEC];
    if (VEC == 4) {
      const float4 q = __ldg(reinterpret_cast<const float4*>(x + b * hw + e));
      v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
      if (seg) {
        if constexpr (sizeof(T) == 8) {
          const longlong2 s0 = __ldg(reinterpret_cast<const longlong2*>(seg + b * hw + e));
          const longlong2 s1 = __ldg(reinterpret_cast<const longlong2*>(seg + b * hw + e + 2));
          sg[0] = s0.x; sg[1] = s0.y; sg[2] = s1.x; sg[3] = s1.y;
        } else {
          const uchar4 s0 = __ldg(reinterpret_cast<const uchar4*>(seg + b * hw + e));
          sg[0] = s0.x; sg[1] = s0.y; sg[2] = s0.z; sg[3] = s0.w;
        }
      }
    } else {
      v[0] = x[b * hw + e];
      if (seg) sg[0] = seg[b * hw + e];
    }
    float vm[VEC];
    uint8_t mm[VEC];
    const int r = static_cast<int>(e / W), c0 = static_cast<int>(e % W);  // W % VEC == 0: the VEC pixels share a row
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      bool m = true;
      if (seg) m = sg[k] == label;
      if (use_thr) m = m && (v[k] <= thr);
      vm[k] = m ? v[k] : v[k] * 0.0f;  // x * m with m in {0,1}
      mm[k] = m ? 1 : 0;
      if (vm[k] != 0.0f) {  // image.nonzero() (utils.py:57): nonzero PIXELS, not nonzero mask
        rmin = min(rmin, r); rmax = max(rmax, r); cmin = min(cmin, c0 + k); cmax = max(cmax, c0 + k);
      }
    }
    if (VEC == 4) {
      if (mask) *reinterpret_cast<uchar4*>(mask + b * hw + e) = make_uchar4(mm[0], mm[1], mm[2], mm[3]);
      if (xm) *reinterpret_cast<float4*>(xm + b * hw + e) = make_float4(vm[0], vm[1], vm[2], vm[3]);
    } else {
      if (mask) mask[b * hw + e] = mm[0];
      if (xm) xm[b * hw + e] = vm[0];
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    rmin = min(rmin, __shfl_xor_sync(0xffffffffu, rmin, o));
    cmin = min(cmin, __shfl_xor_sync(0xffffffffu, cmin, o));
    rmax = max(rmax, __shfl_xor_sync(0xffffffffu, rmax, o));
    cmax = max(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
  }
  if ((threadIdx.x & 31) == 0 && rmax >= 0) {
    atomicMin(&bbox[b * 4 + 0], rmin); atomicMin(&bbox[b * 4 + 1], cmin);
    atomicMax(&bbox[b * 4 + 2], rmax); atomicMax(&bbox[b * 4 + 3], cmax);
  }
}

// ---- antialiased bilinear weights (ATen UpSampleKernel.cpp, HelperInterpLinear, align_corners=False) ----
struct AA {
  int lo, n;
  float scale, support, invscale, center;
};
__device__ __forceinline__ AA aa_setup(int in_size, int out_size, int o) {
  AA a;
  a.scale = static_cast<float>(in_size) / static_cast<float>(out_size);
  a.support = a.scale >= 1.0f ? a.scale : 1.0f;
  a.invscale = a.scale >= 1.0f ? 1.0f / a.scale : 1.0f;
  a.center = a.scale * (o + 0.5f);
  a.lo = max(static_cast<int>(a.center - a.support + 0.5f), 0);
  a.n = min(static_cast<int>(a.center + a.support + 0.5f), in_size) - a.lo;
  return a;
}
__device__ __forceinline__ float aa_w(const AA& a, int j) {
  const float t = fabsf((j + a.lo - a.center + 0.5f) * a.invscale);
  return t < 1.0f ? 1.0f - t : 0.0f;
}

static constexpr int kRsTX = 32, kRsTY = 8;   // output tile of one block
static constexpr int kRsMaxTaps = 20;          // taps kept in shared memory (scale factors up to ~9); above: on the fly

// normalised tap weights of output index o, exactly as the scalar formulation computes them (w_j / sum_j w_j in fp32)
__device__ __forceinline__ void aa_fill(int in_size, int out_size, int o, int* lo, int* n, float* w) {
  const AA a = aa_setup(in_size, out_size, o);
  *lo = a.lo; *n = a.n;
  if (a.n > kRsMaxTaps) return;
  float ws = 0.f;
  for (int j = 0; j < a.n; ++j) ws += aa_w(a, j);
  for (int j = 0; j < a.n; ++j) w[j] = ws != 0.f ? aa_w(a, j) / ws : aa_w(a, j);
}

// out[b, 0, r, c] over the destination window, gray = .2989 R + .587 G + .114 B of src when src_c == 3.
// mode 0: plain resize into dst [B,dst_c,oh,ow] (channels replicated dst_c times) from the src window
//         (bbox rows/cols inclusive, or the whole image when src_bbox == NULL); src_mask (optional, uint8 [B,1,SH,SW])
//         multiplies the source first (the drivers' `c_img * c_m_iris`, …2019.py:66-68)
// mode 1: composite: dst frame [B,1,H,W] in place, window = dst_bbox; frame = mask ? value : frame
__global__ void __launch_bounds__(kRsTX * kRsTY)
resize_aa_kernel(const float* __restrict__ src, int src_c, int SH, int SW, const int32_t* __restrict__ src_bbox,
                 const uint8_t* __restrict__ src_mask, float* __restrict__ dst, int dst_c, int DH, int DW,
                 const int32_t* __restrict__ dst_bbox, const uint8_t* __restrict__ mask, int mode) {
  __shared__ float s_wx[kRsTX][kRsMaxTaps], s_wy[kRsTY][kRsMaxTaps];
  __shared__ int s_xlo[kRsTX], s_xn[kRsTX], s_ylo[kRsTY], s_yn[kRsTY];
  const int b = blockIdx.z;
  int sy0 = 0, sx0 = 0, sh = SH, sw = SW;
  if (src_bbox) {
    sy0 = src_bbox[b * 4 + 0]; sx0 = src_bbox[b * 4 + 1];
    sh = src_bbox[b * 4 + 2] - sy0 + 1; sw = src_bbox[b * 4 + 3] - sx0 + 1;
  }
  int dy0 = 0, dx0 = 0, oh = DH, ow = DW;
  if (dst_bbox) {
    dy0 = dst_bbox[b * 4 + 0]; dx0 = dst_bbox[b * 4 + 1];
    oh = dst_bbox[b * 4 + 2] - dy0 + 1; ow = dst_bbox[b * 4 + 3] - dx0 + 1;
  }
  if (sh <= 0 || sw <= 0 || oh <= 0 || ow <= 0) return;
  const int c_base = blockIdx.x * kRsTX, r_base = blockIdx.y * kRsTY;
  if (c_base >= ow || r_base >= oh) return;  // the grid covers the largest possible window
  const int tx = threadIdx.x % kRsTX, ty = threadIdx.x / kRsTX;
  if (threadIdx.x < kRsTX) {
    if (c_base + threadIdx.x < ow) aa_fill(sw, ow, c_base + threadIdx.x, &s_xlo[threadIdx.x], &s_xn[threadIdx.x], s_wx[threadIdx.x]);
  } else if (threadIdx.x < kRsTX + kRsTY) {
    const int t = threadIdx.x - kRsTX;
    if (r_base + t < oh) aa_fill(sh, oh, r_base + t, &s_ylo[t], &s_yn[t], s_wy[t]);
  }
  __syncthreads();
  const int r = r_base + ty, c = c_base + tx;
  if (r >= oh || c >= ow) return;
  const long o = (static_cast<long>(b) * DH + dy0 + r) * DW + dx0 + c;   // dst_c == 1 addressing (mode 1)
  if (mode == 1 && !mask[o]) return;  // frame * ~m + new * m (…2019.py:125-130): nothing to compute where m == 0
  const long shw = static_cast<long>(SH) * SW;
  const float* sb = src + static_cast<long>(b) * src_c * shw;
  const uint8_t* mb = src_mask ? src_mask + static_cast<long>(b) * shw : nullptr;
  const int xlo = s_xlo[tx], xn = s_xn[tx], ylo = s_ylo[ty], yn = s_yn[ty];
  const bool tab = xn <= kRsMaxTaps && yn <= kRsMaxTaps;
  AA ax, ay;
  float wxs = 0.f, wys = 0.f;
  if (!tab) {  // very large scale factors: weights on the fly (same arithmetic)
    ax = aa_setup(sw, ow, c); ay = aa_setup(sh, oh, r);
    for (int j = 0; j < ax.n; ++j) wxs += aa_w(ax, j);
    for (int j = 0; j < ay.n; ++j) wys += aa_w(ay, j);
  }
  float acc = 0.f;
  for (int jy = 0; jy < yn; ++jy) {
    const long rowoff = static_cast<long>(sy0 + ylo + jy) * SW + sx0 + xlo;
    float t = 0.f;
    for (int jx = 0; jx < xn; ++jx) {
      float v;
      if (src_c == 3) {
        const float R = __ldg(sb + rowoff + jx), G = __ldg(sb + shw + rowoff + jx), Bc = __ldg(sb + 2 * shw + rowoff + jx);
        v = __fadd_rn(__fadd_rn(__fmul_rn(R, 0.2989f), __fmul_rn(G, 0.587f)), __fmul_rn(Bc, 0.114f));
      } else {
        v = __ldg(sb + rowoff + jx);
      }
      if (mb && !mb[rowoff + jx]) v = 0.f;
      const float w = tab ? s_wx[tx][jx] : (wxs != 0.f ? aa_w(ax, jx) / wxs : aa_w(ax, jx));
      t = jx == 0 ? __fmul_rn(v, w) : __fadd_rn(t, __fmul_rn(v, w));
    }
    const float w = tab ? s_wy[ty][jy] : (wys != 0.f ? aa_w(ay, jy) / wys : aa_w(ay, jy));
    acc = jy == 0 ? __fmul_rn(t, w) : __fadd_rn(acc, __fmul_rn(t, w));
  }
  if (mode == 0) {
    for (int ch = 0; ch < dst_c; ++ch)
      dst[((static_cast<long>(b) * dst_c + ch) * DH + dy0 + r) * DW + dx0 + c] = acc;
  } else {
    dst[o] = acc;
  }
}

static int launch_resize(const float* src, int src_c, int SH, int SW, const int32_t* src_bbox, const uint8_t* src_mask,
                         float* dst, int dst_c, int DH, int DW, const int32_t* dst_bbox, const uint8_t* mask, int mode,
                         int B, cudaStream_t s) {
  dim3 grid((DW + kRsTX - 1) / kRsTX, (DH + kRsTY - 1) / kRsTY, B);
  resize_aa_kernel<<<grid, kRsTX * kRsTY, 0, s>>>(src, src_c, SH, SW, src_bbox, src_mask, dst, dst_c, DH, DW, dst_bbox,
                                                  mask, mode);
  ISX_LAUNCH_CHECK();
  return 0;
}

}  // namespace isx

using namespace isx;
static inline cudaStream_t S(isx_stream s) { return reinterpret_cast<cudaStream_t>(s); }

extern "C" int isx_mask_bbox_typed(const float* x, const void* seg, int seg_dtype, int label, int use_threshold, float threshold,
                                   uint8_t* mask, float* xm, int32_t* bbox, int B, int H, int W, isx_stream stream) {
  ISX_REQUIRE(seg_dtype == 0 || seg_dtype == 1, "isx_mask_bbox: seg_dtype %d (0 = int64, 1 = uint8)", seg_dtype);
  ISX_REQUIRE(x && bbox && B > 0 && H > 0 && W > 0, "isx_mask_bbox: bad arguments");
  bbox_init_kernel<<<(B + 127) / 128, 128, 0, S(stream)>>>(bbox, B);
  ISX_LAUNCH_CHECK();
  const long hw = static_cast<long>(H) * W;
  auto al16 = [](const void* p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  const bool u8 = seg_dtype == 1;
  const bool seg_al = u8 ? (reinterpret_cast<uintptr_t>(seg) & 3) == 0 : al16(seg);
  const bool vec = (W % 4 == 0) && al16(x) && seg_al && al16(xm) && (mask == nullptr || (reinterpret_cast<uintptr_t>(mask) & 3) == 0);
  const long items = vec ? hw / 4 : hw;
  // whole waves of 256-thread blocks: 148 SMs x 8 resident blocks, split over the images
  const int bx = static_cast<int>(std::min<long>((items + 255) / 256, std::max<long>(1, static_cast<long>(isx_num_sms()) * 8 / B)));
  dim3 grid(bx, B);
  const int64_t* s64 = static_cast<const int64_t*>(seg);
  const uint8_t* s8 = static_cast<const uint8_t*>(seg);
  if (u8 && vec)
    mask_bbox_kernel<4, uint8_t><<<grid, 256, 0, S(stream)>>>(x, s8, label, use_threshold, threshold, mask, xm, bbox, H, W);
  else if (u8)
    mask_bbox_kernel<1, uint8_t><<<grid, 256, 0, S(stream)>>>(x, s8, label, use_threshold, threshold, mask, xm, bbox, H, W);
  else if (vec)
    mask_bbox_kernel<4, int64_t><<<grid, 256, 0, S(stream)>>>(x, s64, label, use_threshold, threshold, mask, xm, bbox, H, W);
  else
    mask_bbox_kernel<1, int64_t><<<grid, 256, 0, S(stream)>>>(x, s64, label, use_threshold, threshold, mask, xm, bbox, H, W);
  ISX_LAUNCH_CHECK();
  return 0;
}

extern "C" int isx_mask_bbox(const float* x, const int64_t* seg, int label, int use_threshold, float threshold,
                             uint8_t* mask, float* xm, int32_t* bbox, int B, int H, int W, isx_stream stream) {
  return isx_mask_bbox_typed(x, seg, 0, label, use_threshold, threshold, mask, xm, bbox, B, H, W, stream);
}

extern "C" int isx_resize_bilinear_aa(const float* src, int src_c, int SH, int SW, const int32_t* src_bbox, float* dst,
                                      int dst_c, int DH, int DW, int B, isx_stream stream) {
  ISX_REQUIRE(src && dst && (src_c == 1 || src_c == 3) && dst_c >= 1 && B > 0, "isx_resize_bilinear_aa: bad arguments");
  return launch_resize(src, src_c, SH, SW, src_bbox, nullptr, dst, dst_c, DH, DW, nullptr, nullptr, 0, B, S(stream));
}

extern "C" int isx_crop_resize_masked(const float* frames, const uint8_t* mask, const int32_t* bbox, float* dst, int dst_c,
                                      int DH, int DW, int B, int H, int W, isx_stream stream) {
  ISX_REQUIRE(frames && mask && bbox && dst && dst_c >= 1 && B > 0, "isx_crop_resize_masked: bad arguments");
  return launch_resize(frames, 1, H, W, bbox, mask, dst, dst_c, DH, DW, nullptr, nullptr, 0, B, S(stream));
}

extern "C" int isx_composite(const float* new_iris, int src_c, int SH, int SW, float* frames, const uint8_t* mask,
                             const int32_t* bbox, int B, int H, int W, isx_stream stream) {
  ISX_REQUIRE(new_iris && frames && mask && bbox && (src_c == 1 || src_c == 3) && B > 0, "isx_composite: bad arguments");
  return launch_resize(new_iris, src_c, SH, SW, nullptr, nullptr, frames, 1, H, W, bbox, mask, 1, B, S(stream));
}
