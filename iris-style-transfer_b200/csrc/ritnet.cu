// The mask PRODUCER of the hot path on the device (SURVEY.md §8f row 1): the reference's RITnet segmenter,
// models/ritnet/ritnet.py:8-223, called once per eye frame by both drivers (iris_style_transfer_openeds2019.py:155,
// data_preprocessing.py:165) -- there with a CPU round-trip through OpenCV per image (ritnet.py:88-98).
//
//   RITnet_transform (ritnet.py:64-98), bit-exact integer / byte work:
//     u8 = uint8(x * 255) -> gamma table (cv2.LUT + np.uint8) -> CLAHE(clipLimit 1.5, 8x8 tiles) -> normalise table
//     CLAHE restates OpenCV's CLAHE_CalcLut_Body / CLAHE_Interpolation_Body (modules/imgproc/src/clahe.cpp): per-tile
//     histogram (shared-memory atomics), clip + redistribute, cumulative LUT with cvRound, bilinear blend of the four
//     neighbouring tile LUTs in fp32 WITHOUT fma contraction (the CPU code has none), BORDER_REFLECT_101 padding when the
//     frame is not divisible by the tile grid.  Validated against cv2 itself in the tests.
//   DenseNet2D (ritnet.py:100-223), eval mode, fp32:
//     249 225 parameters, every conv has 32 output channels (N = 32 tiles would run the tensor cores issue-bound at a
//     fraction of their rate) and the network runs ONCE per frame against 200-300 closure evaluations of the NST that
//     follows, i.e. < 1 % of the pipeline.  What matters here is that the label map -- index work the mask, the bbox and
//     the crop are derived from -- equals the reference's: with bf16 operands 9-25 labels of a 640x400 frame flip
//     (DESIGN.md §9), in fp32 none do.  So: fp32 CUDA-core direct convolution, NHWC with 32 channels = one 128-byte row
//     per pixel, channel concatenation / nearest up-sampling folded into the operand gather (no cat / interpolate
//     passes), bias + LeakyReLU + BatchNorm in the epilogue, the 1x1 classifier fused with the arg-max.
#include <algorithm>

#include "../../include/isx.h"
#include "isx_common.cuh"

namespace isx {

// ------------------------------------------------------------------------------------------
// RITnet_transform
// ------------------------------------------------------------------------------------------
__global__ void rit_quant_gamma_kernel(const float* __restrict__ x, const uint8_t* __restrict__ gamma, uint8_t* __restrict__ g8,
                                       long n) {
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const float v = __fmul_rn(x[i], 255.0f);                                    // (x * 255)
    const int q = static_cast<int>(v);                                          // .to(torch.uint8): truncation
    g8[i] = gamma[static_cast<uint8_t>(q)];                                     // cv2.LUT + np.uint8
  }
}

struct ClaheGeom {
  int H, W, th, tw, clip;
  float lut_scale, inv_th, inv_tw;
};
static constexpr int kTiles = 8;

__device__ __forceinline__ int reflect101(int i, int n) { return i < n ? i : 2 * (n - 1) - i; }

// one block per (tile, image): histogram -> clip -> redistribute -> cumulative LUT (uint8 [B][64][256])
__global__ void __launch_bounds__(256)
rit_clahe_lut_kernel(const uint8_t* __restrict__ g8, ClaheGeom g, uint8_t* __restrict__ lut) {
  __shared__ int hist[256];
  __shared__ int scan[256];
  __shared__ int s_clipped;
  const int tile = blockIdx.x, b = blockIdx.y;
  const int ty = tile / kTiles, tx = tile % kTiles;
  const int t = threadIdx.x;
  hist[t] = 0;
  if (t == 0) s_clipped = 0;
  __syncthreads();
  const uint8_t* img = g8 + static_cast<long>(b) * g.H * g.W;
  const int area = g.th * g.tw;
  for (int i = t; i < area; i += 256) {
    const int y = reflect101(ty * g.th + i / g.tw, g.H), x = reflect101(tx * g.tw + i % g.tw, g.W);
    atomicAdd(&hist[img[static_cast<long>(y) * g.W + x]], 1);
  }
  __syncthreads();
  int h = hist[t];
  if (g.clip > 0) {
    if (h > g.clip) { atomicAdd(&s_clipped, h - g.clip); h = g.clip; }
    __syncthreads();
    const int clipped = s_clipped;
    const int batch = clipped / 256;
    int residual = clipped - batch * 256;
    h += batch;
    if (residual != 0) {
      const int step = max(256 / residual, 1);
      if (t % step == 0 && t / step < residual) h += 1;
    }
  }
  // inclusive scan of the 256 bins
  scan[t] = h;
  __syncthreads();
  for (int o = 1; o < 256; o <<= 1) {
    const int v = t >= o ? scan[t - o] : 0;
    __syncthreads();
    scan[t] += v;
    __syncthreads();
  }
  const int r = __float2int_rn(__fmul_rn(static_cast<float>(scan[t]), g.lut_scale));   // saturate_cast<uchar>(sum * lutScale)
  lut[(static_cast<long>(b) * kTiles * kTiles + tile) * 256 + t] = static_cast<uint8_t>(min(max(r, 0), 255));
}

// bilinear blend of the four neighbouring tile LUTs, then the ToDtype/Normalize table -> fp32 network input
__global__ void __launch_bounds__(256)
rit_clahe_interp_kernel(const uint8_t* __restrict__ g8, const uint8_t* __restrict__ lut, const float* __restrict__ norm,
                        ClaheGeom g, float* __restrict__ out) {
  const int b = blockIdx.y;
  const long hw = static_cast<long>(g.H) * g.W;
  const uint8_t* L = lut + static_cast<long>(b) * kTiles * kTiles * 256;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < hw; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int y = static_cast<int>(i / g.W), x = static_cast<int>(i % g.W);
    const float txf = __fsub_rn(__fmul_rn(static_cast<float>(x), g.inv_tw), 0.5f);
    const float tyf = __fsub_rn(__fmul_rn(static_cast<float>(y), g.inv_th), 0.5f);
    int tx1 = static_cast<int>(floorf(txf)), ty1 = static_cast<int>(floorf(tyf));
    const float xa = __fsub_rn(txf, static_cast<float>(tx1)), ya = __fsub_rn(tyf, static_cast<float>(ty1));
    const float xa1 = __fsub_rn(1.0f, xa), ya1 = __fsub_rn(1.0f, ya);
    const int tx2 = min(tx1 + 1, kTiles - 1), ty2 = min(ty1 + 1, kTiles - 1);
    tx1 = max(tx1, 0); ty1 = max(ty1, 0);
    const int v = g8[b * hw + i];
    const float p11 = L[(ty1 * kTiles + tx1) * 256 + v], p12 = L[(ty1 * kTiles + tx2) * 256 + v];
    const float p21 = L[(ty2 * kTiles + tx1) * 256 + v], p22 = L[(ty2 * kTiles + tx2) * 256 + v];
    const float top = __fadd_rn(__fmul_rn(p11, xa1), __fmul_rn(p12, xa));
    const float bot = __fadd_rn(__fmul_rn(p21, xa1), __fmul_rn(p22, xa));
    const float res = __fadd_rn(__fmul_rn(top, ya1), __fmul_rn(bot, ya));
    const int r = min(max(__float2int_rn(res), 0), 255);
    out[b * hw + i] = norm[r];
  }
}

// ------------------------------------------------------------------------------------------
// DenseNet2D: direct fp32 convolution over up to three concatenated NHWC sources -> 32 channels
// ------------------------------------------------------------------------------------------
struct RitSrc {
  const float* p;  // [B, H >> up, W >> up, C]
  int C;
  int up;          // 1: nearest 2x up-sampling folded into the gather (F.interpolate(scale_factor=2), ritnet.py:152)
};

static constexpr int kRtTW = 32, kRtTH = 16, kRtCh = 8;

template <int KS>
__global__ void __launch_bounds__(256, 2)
rit_conv_kernel(RitSrc s0, RitSrc s1, RitSrc s2, int nsrc, int cin_total, const float* __restrict__ w,
                const float* __restrict__ bias, int act, const float* __restrict__ bn_scale,
                const float* __restrict__ bn_shift, float* __restrict__ out, int H, int W) {
  constexpr int R = KS / 2;
  constexpr int PW = kRtTW + 2 * R, PH = kRtTH + 2 * R;
  __shared__ float s_in[kRtCh][PH * PW];                       // channel-major patch: conflict-free row reads
  __shared__ __align__(16) float s_w[KS * KS][kRtCh][32];
  const int b = blockIdx.z;
  const int x0 = blockIdx.x * kRtTW, y0 = blockIdx.y * kRtTH;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // pixels (tx, ty) and (tx, ty + 8) of the tile
  float acc0[32], acc1[32];
#pragma unroll
  for (int o = 0; o < 32; ++o) acc0[o] = acc1[o] = 0.f;
  int cin_off = 0;
  for (int si = 0; si < nsrc; ++si) {
    const RitSrc S = si == 0 ? s0 : (si == 1 ? s1 : s2);
    const int Hs = S.up ? H >> 1 : H, Ws = S.up ? W >> 1 : W;
    for (int c0 = 0; c0 < S.C; c0 += kRtCh) {
      const int cc = min(kRtCh, S.C - c0);
      __syncthreads();
      for (int i = threadIdx.x; i < PH * PW; i += 256) {
        const int gy = y0 + i / PW - R, gx = x0 + i % PW - R;
        float v[kRtCh];
#pragma unroll
        for (int k = 0; k < kRtCh; ++k) v[k] = 0.f;
        if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
          const int sy = S.up ? gy >> 1 : gy, sx = S.up ? gx >> 1 : gx;
          const float* q = S.p + ((static_cast<long>(b) * Hs + sy) * Ws + sx) * S.C + c0;
          if (cc == kRtCh) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(q)), c4 = __ldg(reinterpret_cast<const float4*>(q + 4));
            v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = c4.x; v[5] = c4.y; v[6] = c4.z; v[7] = c4.w;
          } else {
            for (int k = 0; k < cc; ++k) v[k] = __ldg(q + k);
          }
        }
#pragma unroll
        for (int k = 0; k < kRtCh; ++k) s_in[k][i] = v[k];
      }
      for (int i = threadIdx.x; i < KS * KS * kRtCh * 8; i += 256) {
        const int tap = i / (kRtCh * 8), c = (i >> 3) % kRtCh, o4 = i & 7;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c < cc) v = __ldg(reinterpret_cast<const float4*>(w + (static_cast<long>(tap) * cin_total + cin_off + c0 + c) * 32) + o4);
        reinterpret_cast<float4*>(&s_w[tap][c][0])[o4] = v;
      }
      __syncthreads();
#pragma unroll 1
      for (int tap = 0; tap < KS * KS; ++tap) {
        const int dy = tap / KS, dx = tap % KS;
        const int i0 = (ty + dy) * PW + tx + dx, i1 = (ty + 8 + dy) * PW + tx + dx;
#pragma unroll
        for (int c = 0; c < kRtCh; ++c) {
          const float a0 = s_in[c][i0], a1 = s_in[c][i1];
#pragma unroll
          for (int o4 = 0; o4 < 8; ++o4) {
            const float4 wv = reinterpret_cast<const float4*>(&s_w[tap][c][0])[o4];
            acc0[4 * o4 + 0] = fmaf(a0, wv.x, acc0[4 * o4 + 0]); acc0[4 * o4 + 1] = fmaf(a0, wv.y, acc0[4 * o4 + 1]);
            acc0[4 * o4 + 2] = fmaf(a0, wv.z, acc0[4 * o4 + 2]); acc0[4 * o4 + 3] = fmaf(a0, wv.w, acc0[4 * o4 + 3]);
            acc1[4 * o4 + 0] = fmaf(a1, wv.x, acc1[4 * o4 + 0]); acc1[4 * o4 + 1] = fmaf(a1, wv.y, acc1[4 * o4 + 1]);
            acc1[4 * o4 + 2] = fmaf(a1, wv.z, acc1[4 * o4 + 2]); acc1[4 * o4 + 3] = fmaf(a1, wv.w, acc1[4 * o4 + 3]);
          }
        }
      }
    }
    cin_off += S.C;
  }
  // epilogue: bias -> LeakyReLU(0.01) -> BatchNorm (eval: per-channel affine), 128-byte rows
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int gy = y0 + ty + 8 * half, gx = x0 + tx;
    if (gy >= H || gx >= W) continue;
    float* dst = out + ((static_cast<long>(b) * H + gy) * W + gx) * 32;
#pragma unroll
    for (int o4 = 0; o4 < 8; ++o4) {
      float r[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int o = 4 * o4 + k;
        float v = (half ? acc1[o] : acc0[o]) + __ldg(bias + o);
        if (act) v = v > 0.f ? v : v * 0.01f;
        if (bn_scale) v = fmaf(v, __ldg(bn_scale + o), __ldg(bn_shift + o));
        r[k] = v;
      }
      reinterpret_cast<float4*>(dst)[o4] = make_float4(r[0], r[1], r[2], r[3]);
    }
  }
}

// AvgPool2d(2) on NHWC-32 (ritnet.py:108,119-120)
__global__ void rit_avgpool_kernel(const float* __restrict__ in, float* __restrict__ out, int B, int H, int W) {
  const int Ho = H >> 1, Wo = W >> 1;
  const long n4 = static_cast<long>(B) * Ho * Wo * 8;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n4; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int c4 = static_cast<int>(i & 7);
    const long p = i >> 3;
    const int xo = static_cast<int>(p % Wo), yo = static_cast<int>((p / Wo) % Ho), b = static_cast<int>(p / (static_cast<long>(Wo) * Ho));
    const float4* s = reinterpret_cast<const float4*>(in + ((static_cast<long>(b) * H + 2 * yo) * W + 2 * xo) * 32) + c4;
    const float4 a = __ldg(s), c = __ldg(s + 8), d = __ldg(s + static_cast<long>(W) * 8), e = __ldg(s + static_cast<long>(W) * 8 + 8);
    reinterpret_cast<float4*>(out)[i] = make_float4((a.x + c.x + d.x + e.x) * 0.25f, (a.y + c.y + d.y + e.y) * 0.25f,
                                                    (a.z + c.z + d.z + e.z) * 0.25f, (a.w + c.w + d.w + e.w) * 0.25f);
  }
}

// out_conv1 (1x1, 32 -> 4, ritnet.py:195) fused with `_, x = x.max(1)` (ritnet.py:55): first maximal class wins.
// T = int64_t (the reference's dtype) or uint8_t (1 B per pixel for the consumers that read uint8 maps natively).
template <typename T>
__global__ void rit_classify_kernel(const float* __restrict__ x9, const float* __restrict__ w, const float* __restrict__ bias,
                                    T* __restrict__ labels, float* __restrict__ logits, long hw, long npix) {
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < npix; i += static_cast<long>(gridDim.x) * blockDim.x) {
    float l[4] = {__ldg(bias), __ldg(bias + 1), __ldg(bias + 2), __ldg(bias + 3)};
    const float4* s = reinterpret_cast<const float4*>(x9 + i * 32);
#pragma unroll
    for (int c4 = 0; c4 < 8; ++c4) {
      const float4 v = __ldg(s + c4);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float4 wk = __ldg(reinterpret_cast<const float4*>(w + k * 32) + c4);
        l[k] = fmaf(v.x, wk.x, l[k]); l[k] = fmaf(v.y, wk.y, l[k]); l[k] = fmaf(v.z, wk.z, l[k]); l[k] = fmaf(v.w, wk.w, l[k]);
      }
    }
    int best = 0;
#pragma unroll
    for (int k = 1; k < 4; ++k) if (l[k] > l[best]) best = k;
    labels[i] = static_cast<T>(best);
    if (logits) {
      const long b = i / hw, p = i - b * hw;
#pragma unroll
      for (int k = 0; k < 4; ++k) logits[(b * 4 + k) * hw + p] = l[k];
    }
  }
}

// ------------------------------------------------------------------------------------------
// parameter blob: fixed architecture, offsets in floats (the Python side packs in the same order)
// ------------------------------------------------------------------------------------------
struct RitConv { long w, b; int ks, cin; };
struct RitPlan {
  RitConv down[5][5];   // conv1, conv21, conv22, conv31, conv32
  long bn_scale[5], bn_shift[5];
  RitConv up[4][4];     // conv11, conv12, conv21, conv22
  long out_w, out_b;
  long total;
};

static RitPlan make_plan() {
  RitPlan P;
  long off = 0;
  auto conv = [&](int ks, int cin) { RitConv c; c.ks = ks; c.cin = cin; c.w = off; off += static_cast<long>(ks) * ks * cin * 32; c.b = off; off += 32; return c; };
  for (int k = 0; k < 5; ++k) {
    const int cin = k == 0 ? 1 : 32;
    P.down[k][0] = conv(3, cin); P.down[k][1] = conv(1, cin + 32); P.down[k][2] = conv(3, 32);
    P.down[k][3] = conv(1, cin + 64); P.down[k][4] = conv(3, 32);
    P.bn_scale[k] = off; off += 32; P.bn_shift[k] = off; off += 32;
  }
  for (int k = 0; k < 4; ++k) {
    P.up[k][0] = conv(1, 64); P.up[k][1] = conv(3, 32); P.up[k][2] = conv(1, 96); P.up[k][3] = conv(3, 32);
  }
  P.out_w = off; off += 4 * 32; P.out_b = off; off += 4;
  P.total = off;
  return P;
}

static int launch_conv(const RitConv& c, const float* params, RitSrc s0, RitSrc s1, RitSrc s2, int nsrc, int act,
                       const float* bn_scale, const float* bn_shift, float* out, int B, int H, int W, cudaStream_t s) {
  dim3 grid((W + kRtTW - 1) / kRtTW, (H + kRtTH - 1) / kRtTH, B);
  if (c.ks == 3)
    rit_conv_kernel<3><<<grid, 256, 0, s>>>(s0, s1, s2, nsrc, c.cin, params + c.w, params + c.b, act, bn_scale, bn_shift, out, H, W);
  else
    rit_conv_kernel<1><<<grid, 256, 0, s>>>(s0, s1, s2, nsrc, c.cin, params + c.w, params + c.b, act, bn_scale, bn_shift, out, H, W);
  ISX_LAUNCH_CHECK();
  return 0;
}

}  // namespace isx

using namespace isx;
static inline cudaStream_t S(isx_stream s) { return reinterpret_cast<cudaStream_t>(s); }

extern "C" int64_t isx_ritnet_param_floats(void) { return make_plan().total; }

static size_t rit_align(size_t v) { return (v + 255) & ~size_t(255); }

extern "C" int64_t isx_ritnet_workspace_bytes(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0 || H % 16 || W % 16) return -1;
  size_t off = 0;
  const size_t hw = static_cast<size_t>(H) * W;
  off += rit_align(B * hw);                       // gamma-corrected uint8 frames
  off += rit_align(static_cast<size_t>(B) * 64 * 256);  // CLAHE LUTs
  off += rit_align(B * hw * 4);                   // network input
  for (int l = 0; l < 5; ++l) off += 5 * rit_align(static_cast<size_t>(B) * (H >> l) * (W >> l) * 32 * 4);
  return static_cast<int64_t>(off);
}

namespace {
struct RitPre { uint8_t* g8; uint8_t* lut; };
// RITnet_transform for a batch: x [B,1,H,W] -> out fp32 [B,1,H,W]; scratch g8 (B*H*W bytes) and lut (B*64*256 bytes)
int run_transform(const float* x, const uint8_t* gamma_lut, const float* norm_lut, uint8_t* g8, uint8_t* lut, float* out,
                  int B, int H, int W, cudaStream_t s) {
  const size_t hw = static_cast<size_t>(H) * W;
  const long n = static_cast<long>(B) * hw;
  const int blocks = static_cast<int>(std::min<long>((n + 255) / 256, static_cast<long>(isx_num_sms()) * 16));
  rit_quant_gamma_kernel<<<blocks, 256, 0, s>>>(x, gamma_lut, g8, n);
  ISX_LAUNCH_CHECK();
  ClaheGeom g;
  g.H = H; g.W = W;
  int He = H, We = W;
  if (W % kTiles != 0 || H % kTiles != 0) { He = H + (kTiles - H % kTiles); We = W + (kTiles - W % kTiles); }
  g.th = He / kTiles; g.tw = We / kTiles;
  const int area = g.th * g.tw;
  g.lut_scale = 255.0f / static_cast<float>(area);
  g.clip = std::max(static_cast<int>(1.5 * area / 256), 1);   // clipLimit 1.5 (ritnet.py:71)
  g.inv_th = 1.0f / static_cast<float>(g.th); g.inv_tw = 1.0f / static_cast<float>(g.tw);
  rit_clahe_lut_kernel<<<dim3(kTiles * kTiles, B), 256, 0, s>>>(g8, g, lut);
  ISX_LAUNCH_CHECK();
  rit_clahe_interp_kernel<<<dim3(static_cast<unsigned>(std::min<long>((hw + 255) / 256, static_cast<long>(isx_num_sms()) * 8)), B), 256, 0, s>>>(g8, lut, norm_lut, g, out);
  ISX_LAUNCH_CHECK();
  return 0;
}
}  // namespace

extern "C" int64_t isx_ritnet_transform_workspace_bytes(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return -1;
  return static_cast<int64_t>(rit_align(static_cast<size_t>(B) * H * W) + rit_align(static_cast<size_t>(B) * 64 * 256));
}

extern "C" int isx_ritnet_transform(const float* x, const uint8_t* gamma_lut, const float* norm_lut, void* workspace, float* out,
                                    int B, int H, int W, isx_stream stream) {
  ISX_REQUIRE(x && gamma_lut && norm_lut && workspace && out && B > 0 && H >= 8 && W >= 8, "isx_ritnet_transform: bad arguments");
  char* ws = static_cast<char*>(workspace);
  return run_transform(x, gamma_lut, norm_lut, reinterpret_cast<uint8_t*>(ws),
                       reinterpret_cast<uint8_t*>(ws + rit_align(static_cast<size_t>(B) * H * W)), out, B, H, W, S(stream));
}

extern "C" int isx_ritnet_forward_typed(const float* x, const float* params, const uint8_t* gamma_lut, const float* norm_lut,
                                        void* workspace, void* labels, int label_dtype, float* logits, int B, int H, int W,
                                        isx_stream stream) {
  ISX_REQUIRE(label_dtype == 0 || label_dtype == 1, "isx_ritnet_forward: label_dtype %d (0 = int64, 1 = uint8)", label_dtype);
  ISX_REQUIRE(x && params && gamma_lut && norm_lut && workspace && labels, "isx_ritnet_forward: null pointer");
  ISX_REQUIRE(B > 0 && H >= 16 && W >= 16 && H % 16 == 0 && W % 16 == 0,
              "isx_ritnet_forward: frame %dx%d must be a positive multiple of 16 in both dimensions (four 2x2 poolings and "
              "the skip concatenations of DenseNet2D, ritnet.py:209-218)", H, W);
  cudaStream_t s = S(stream);
  const RitPlan P = make_plan();
  char* ws = static_cast<char*>(workspace);
  const size_t hw = static_cast<size_t>(H) * W;
  size_t off = 0;
  uint8_t* g8 = reinterpret_cast<uint8_t*>(ws + off); off += rit_align(B * hw);
  uint8_t* lut = reinterpret_cast<uint8_t*>(ws + off); off += rit_align(static_cast<size_t>(B) * 64 * 256);
  float* xin = reinterpret_cast<float*>(ws + off); off += rit_align(B * hw * 4);
  float* buf[5][5];  // per level: pooled input, a, t, b, X (skip)
  for (int l = 0; l < 5; ++l)
    for (int k = 0; k < 5; ++k) { buf[l][k] = reinterpret_cast<float*>(ws + off); off += rit_align(static_cast<size_t>(B) * (H >> l) * (W >> l) * 32 * 4); }

  // ---- RITnet_transform ----
  const long n = static_cast<long>(B) * hw;
  if (int rc = run_transform(x, gamma_lut, norm_lut, g8, lut, xin, B, H, W, s)) return rc;

  // ---- DenseNet2D ----
  RitSrc none{nullptr, 0, 0};
  for (int l = 0; l < 5; ++l) {   // down blocks (ritnet.py:118-135)
    const int h = H >> l, w = W >> l;
    RitSrc in;
    if (l == 0) {
      in = RitSrc{xin, 1, 0};
    } else {
      const long n4 = static_cast<long>(B) * h * w * 8;
      rit_avgpool_kernel<<<static_cast<int>(std::min<long>((n4 + 255) / 256, static_cast<long>(isx_num_sms()) * 16)), 256, 0, s>>>(buf[l - 1][4], buf[l][0], B, H >> (l - 1), W >> (l - 1));
      ISX_LAUNCH_CHECK();
      in = RitSrc{buf[l][0], 32, 0};
    }
    RitSrc a{buf[l][1], 32, 0}, t{buf[l][2], 32, 0}, bb{buf[l][3], 32, 0};
    if (int rc = launch_conv(P.down[l][0], params, in, none, none, 1, 1, nullptr, nullptr, buf[l][1], B, h, w, s)) return rc;   // x1
    if (int rc = launch_conv(P.down[l][1], params, in, a, none, 2, 0, nullptr, nullptr, buf[l][2], B, h, w, s)) return rc;      // conv21(x21)
    if (int rc = launch_conv(P.down[l][2], params, t, none, none, 1, 1, nullptr, nullptr, buf[l][3], B, h, w, s)) return rc;    // x22
    if (int rc = launch_conv(P.down[l][3], params, in, a, bb, 3, 0, nullptr, nullptr, buf[l][2], B, h, w, s)) return rc;        // conv31(x31)
    if (int rc = launch_conv(P.down[l][4], params, t, none, none, 1, 1, params + P.bn_scale[l], params + P.bn_shift[l], buf[l][4], B, h, w, s)) return rc;
  }
  const float* prev = buf[4][4];
  for (int k = 0; k < 4; ++k) {   // up blocks (ritnet.py:151-162); level 3 .. 0
    const int l = 3 - k, h = H >> l, w = W >> l;
    RitSrc up{prev, 32, 1}, skip{buf[l][4], 32, 0}, t{buf[l][2], 32, 0}, d{buf[l][1], 32, 0};
    if (int rc = launch_conv(P.up[k][0], params, up, skip, none, 2, 0, nullptr, nullptr, buf[l][2], B, h, w, s)) return rc;     // conv11
    if (int rc = launch_conv(P.up[k][1], params, t, none, none, 1, 1, nullptr, nullptr, buf[l][1], B, h, w, s)) return rc;      // x1
    if (int rc = launch_conv(P.up[k][2], params, up, skip, d, 3, 0, nullptr, nullptr, buf[l][2], B, h, w, s)) return rc;        // conv21
    if (int rc = launch_conv(P.up[k][3], params, t, none, none, 1, 1, nullptr, nullptr, buf[l][3], B, h, w, s)) return rc;      // out
    prev = buf[l][3];
  }
  const int cblocks = static_cast<int>(std::min<long>((n + 255) / 256, static_cast<long>(isx_num_sms()) * 16));
  if (label_dtype == 1)
    rit_classify_kernel<uint8_t><<<cblocks, 256, 0, s>>>(prev, params + P.out_w, params + P.out_b, static_cast<uint8_t*>(labels),
                                                         logits, static_cast<long>(hw), n);
  else
    rit_classify_kernel<int64_t><<<cblocks, 256, 0, s>>>(prev, params + P.out_w, params + P.out_b, static_cast<int64_t*>(labels),
                                                         logits, static_cast<long>(hw), n);
  ISX_LAUNCH_CHECK();
  return 0;
}

extern "C" int isx_ritnet_forward(const float* x, const float* params, const uint8_t* gamma_lut, const float* norm_lut,
                                  void* workspace, int64_t* labels, float* logits, int B, int H, int W, isx_stream stream) {
  return isx_ritnet_forward_typed(x, params, gamma_lut, norm_lut, workspace, labels, 0, logits, B, H, W, stream);
}
